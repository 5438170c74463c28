"""Full-size parity: candidates sampled from INSIDE the BASELINE.json batches (config 2 at 4096,
config 3 at 256 fields x 180 headings, config 5 at 8192 candidates) are compared field by field
with the CPU oracle (oracle.batch.evaluate_candidate), so that a defect that depends on the batch
position, on the coverage de-duplication's hash table at scale or on the plan kernel's launch tiers
cannot hide behind GPU-vs-GPU comparisons.  The oracle calls of one test run in a process pool.

Tolerances as in test_gpu_parity.py: counts bit-exact, FP64 sums rtol 1e-9, points and speeds 1e-9
(north_star asks 1e-4 m / 1e-4 m/s).
"""
import multiprocessing as mp
import os

import numpy as np
import pytest

from benchmarks import workloads as wl

pytestmark = pytest.mark.gpu

TIGHT = 1e-9


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


def _oracle_one(job):
    from oracle import batch as ob, ref_planner as rp
    (verts, R, heading, corner, obst, h), coverage, keep = job[:3]
    veh = rp.VehicleParams(**(job[3] if len(job) > 3 else {}))
    extra = job[4] if len(job) > 4 else {}
    return ob.evaluate_candidate(verts, veh, R=R, heading=heading, start_corner=corner, obstacles=obst,
                                 grid_h=h, coverage=coverage, keep_paths=keep, **extra)


def oracle_many(jobs):
    """[(oracle_args, coverage, keep_paths[, vehicle fields[, evaluate_candidate keywords]])] -> oracle records, in a
    fork pool (the children never touch CUDA).  The vehicle fields are a dict of rp.VehicleParams fields (the
    defaults when absent); the keywords are e.g. turn_model / clothoid_share."""
    from oracle import raster
    raster.build()
    n = min(len(jobs), os.cpu_count() or 1)
    if n <= 1:
        return [_oracle_one(j) for j in jobs]
    with mp.get_context("fork").Pool(n) as pool:
        return pool.map(_oracle_one, jobs, chunksize=1)


def summary_vs_oracle(s, o, coverage=True):
    assert int(s["status"]) == o["status"]
    if o["status"]:
        return
    for k in ("n_passes", "n_loops", "n_main", "n_head", "n_accel_viol", "n_boundary_viol", "n_obstacle_viol"):
        assert int(s[k]) == int(o[k]), (k, int(s[k]), o[k])
    for k in ("len_main", "len_head", "time_main", "time_head", "time_main_pre", "time_head_pre",
              "max_curvature", "max_lateral_accel", "max_jump"):
        np.testing.assert_allclose(float(s[k]), o[k], rtol=1e-9, atol=1e-12, err_msg=k)
    if coverage:
        assert int(s["corner_g"]) == o["corner_g"]
        assert list(map(int, s["corner_before"])) == o["corner_before"]
        assert list(map(int, s["corner_after"])) == o["corner_after"]
        assert (int(s["cov_total"]), int(s["cov_cells"])) == (o["cov_total"], o["cov_cells"])


def sample_indices(n, k, seed, extra=()):
    rng = np.random.default_rng(seed)
    idx = set(int(i) for i in rng.choice(n, size=min(k, n), replace=False))
    idx.update((0, n - 1))
    idx.update(int(i) for i in extra if 0 <= int(i) < n)
    return sorted(idx)


def test_config2_full_batch_sampled_vs_oracle(fc):
    """Config 2 at full size, paths materialised: 40 candidates from inside the 4096 (first, last, seeded random
    positions, the knife-edge radii of SURVEY.md App. A Q17 spliced in, members of every coverage
    de-duplication group that are NOT its representative) against the oracle, every summary field, paths
    and speeds; the batch argmin against numpy on the oracle-checked cost column."""
    w = wl.c2(1)
    cands = {k: v.copy() for k, v in w.cands.items()}
    cands["R"][4 * 100:4 * 100 + 4] = 7.2       # FP64 knife edges inside the batch (Q17)
    cands["R"][4 * 777:4 * 777 + 4] = 9.6
    cands["R"][4 * 901:4 * 901 + 4] = 6.4
    res = fc.plan_batch(w.fields, fc.VehicleParams(), cands, obstacles=w.obstacles, outputs="paths", grid_h=w.grid_h)
    assert len(res.summary) == 4096 and (res.summary["status"] == 0).all()
    # start corners 1-3 share the corner windows of start corner 0 (de-duplicated part 0)
    idx = sample_indices(4096, 30, 2024, extra=(401, 402, 403, 4 * 777 + 1, 4 * 901 + 3, 4 * 511 + 2, 4095 - 1))
    w2 = wl.Workload(w.name, w.text, w.fields, cands, w.obstacles, w.grid_h, w.outputs)
    recs = oracle_many([(w2.oracle_args(i), True, True) for i in idx])
    worst_p = worst_s = 0.0
    for i, o in zip(idx, recs):
        summary_vs_oracle(res.summary[i], o)
        p, s, _ = res.path(i)
        assert p.shape == o["path"].shape
        worst_p = max(worst_p, float(np.abs(p - o["path"]).max()))
        worst_s = max(worst_s, float(np.abs(s - o["speeds"]).max()))
    assert worst_p <= TIGHT and worst_s <= TIGHT, (worst_p, worst_s)
    cost = res.summary["len_main"] + res.summary["len_head"]
    assert int(res.best_cand[0]) == int(np.argmin(cost)) and res.best_cost[0] == cost.min()


def test_config3_256_fields_x_180_headings_sampled_vs_oracle(fc):
    """Config 3 at 256 fields x 180 headings (46 080 candidates, summary only, coverage de-duplicated over
    the headings, three plan-length tiers): sampled candidates — random positions, the shortest and the
    longest plan, plans next to the length quantiles where the launch tiers change — against the oracle;
    the per-field argmin of two whole fields against the oracle's costs."""
    w = wl.c3(1, fields_per_gpu=256)
    res = fc.plan_batch(w.fields, fc.VehicleParams(), w.cands, outputs="summary", grid_h=w.grid_h)
    s = res.summary
    B = len(s)
    assert B == 256 * 180
    n = (s["n_main"] + s["n_head"]).astype(np.int64)
    order = np.argsort(n, kind="stable")
    extra = [order[0], order[-1]] + [order[int(q * (B - 1))] for q in (0.25, 0.5, 0.75, 0.9, 0.99)]
    # within a field the 180 headings share one coverage result: check non-representatives too
    extra += [5 * 180 + 179, 77 * 180 + 1, 255 * 180 + 90]
    idx = sample_indices(B, 26, 7, extra=extra)
    recs = oracle_many([(w.oracle_args(i), True, False) for i in idx])
    n_ok = 0
    for i, o in zip(idx, recs):
        summary_vs_oracle(s[i], o)
        n_ok += o["status"] == 0
    assert n_ok >= 20
    # per-field argmin over the 180 headings: the oracle's costs of two whole fields
    cost = s["len_main"] + s["len_head"]
    for f in (3, 200):
        sl = slice(f * 180, (f + 1) * 180)
        fo = oracle_many([(w.oracle_args(i), False, False) for i in range(sl.start, sl.stop)])
        oc = np.array([(o["len_main"] + o["len_head"]) if o["status"] == 0 else np.inf for o in fo])
        valid = s["status"][sl] == 0
        assert np.array_equal(valid, np.isfinite(oc))
        np.testing.assert_allclose(cost[sl][valid], oc[valid], rtol=1e-9)
        srt = np.sort(oc)
        if srt[1] - srt[0] > 1e-6:       # a unique minimum: the winner must be the oracle's
            assert int(res.best_cand[f]) == f * 180 + int(np.argmin(oc))
        assert int(res.best_cand[f]) == f * 180 + int(np.argmin(np.where(valid, cost[sl], np.inf)))
    # every field's winner equals numpy's argmin of the (oracle-checked) cost column
    c2d = np.where(s["status"] == 0, cost, np.inf).reshape(256, 180)
    want = np.where(np.isfinite(c2d.min(1)), np.arange(256) * 180 + c2d.argmin(1), -1)
    assert np.array_equal(res.best_cand, want)


def test_config5_8192_candidates_sampled_vs_oracle(fc):
    """Config 5 (2 km x 1 km, h = 0.05 m) at one GPU's shard size, 8192 candidates: 32 sampled candidates
    against the oracle for everything but coverage, 10 of them including the 19-million-cell band raster
    (22 s each on one core, hence the process pool)."""
    w = wl.c5(1)
    res = fc.plan_batch(w.fields, fc.VehicleParams(), w.cands, outputs="summary", grid_h=w.grid_h)
    s = res.summary
    assert len(s) == 8192 and (s["status"] == 0).all()
    idx = sample_indices(8192, 30, 55)
    with_cov = set(idx[::3][:10])
    recs = oracle_many([(w.oracle_args(i), i in with_cov, False) for i in idx])
    for i, o in zip(idx, recs):
        summary_vs_oracle(s[i], o, coverage=i in with_cov)
    # the band of a 2000 x 1000 field at 0.05 m in closed form; identical for the four start corners
    R = w.cands["R"]
    tot = s["cov_total"].reshape(-1, 4)
    assert (tot == tot[:, :1]).all()
    cost = s["len_main"] + s["len_head"]
    assert int(res.best_cand[0]) == int(np.argmin(cost))
    assert (s["corner_g"] == (2 * R / 0.1).astype(int)).all()


def test_reference_coverage_values_of_the_fixtures(fc, golden_dir):
    """The reference values stored in the fixtures that no other test reads: `coverage_rate` of the
    headland (mlp3:1357-1371, the stand-in's numeric area, D2) against the integer raster (D5) and the
    corner-grid averages of verify_all_corners_coverage (mlp3:1573-1578)."""
    import glob
    import json
    for path in sorted(glob.glob(os.path.join(golden_dir, "ref_*.npz"))):
        z = np.load(path)
        meta = json.loads(str(z["meta"]))
        kw = dict(meta["planner"])
        for k in ("start_point", "end_point"):
            if kw.get(k) is not None:
                kw[k] = tuple(kw[k])
        if kw.get("field_vertices") is not None:
            kw["field_vertices"] = [tuple(v) for v in kw["field_vertices"]]
        pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(**meta["vehicle"]), **kw)
        r = pl.plan_complete_coverage()
        got = r["headland"]["stats"]["coverage_rate"]
        # observed: <= 2.5e-5 on the rectangles, 1.3e-4 on the sheared field (0.1 m cells along slanted edges)
        assert abs(got - float(z["coverage_rate_sampled"])) <= 2e-4, (os.path.basename(path), got)
        if "corner_avg" in z.files:
            cov = pl.verify_all_corners_coverage(r["headland"])
            ours = [cov["avg_coverage_before"], cov["avg_coverage_after"], cov["avg_improvement"]]
            # float64 contains() of the stand-in vs the exact fixed-point predicate: <= 2 cells of g^2 per corner
            g2 = float(int(2 * meta["vehicle"]["min_turn_radius"] / 0.1) ** 2)
            np.testing.assert_allclose(ours, z["corner_avg"], rtol=0, atol=100.0 * 2 / g2 + 1e-9)
