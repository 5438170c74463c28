"""GPU tests of the launch variants that the kernels select from a size, and of the per-point curvature outputs.

Many entry points pick a kernel instance from a path length, a batch size or a grid size: the caller-supplied-path
kernels run in up to three shared-memory tiers plus an HBM-staged kernel, the prefix sum of the path offsets goes
multi-tile beyond 4096 candidates, the per-field argmin switches kernels at 16384 candidates or fields, the coverage
kernel runs one CTA per candidate or a persistent work list, and the window raster splits large windows into row
tiles and long polylines into point chunks.  Every test here builds inputs that sit on both sides of such a switch
and compares the result with the float64 / integer oracle (``oracle/``), or, where two variants must agree, checks
that they are byte-identical.  Output buffers are filled with NaN bytes before each call, so an output the kernel
never writes cannot pass by accident.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]
OBST2 = [[(200, 80), (250, 80), (250, 120), (200, 120)], [(350, 140), (380, 140), (380, 170), (350, 170)]]
PARA = [(100, 50), (600, 120), (640, 330), (140, 260)]
SMALL = [(0, 0), (60, 0), (60, 45), (0, 45)]
DEAD = [(0, 0), (12, 0), (12, 9), (0, 9)]           # inset empty at every R >= 4.5: no valid candidate
TIGHT = 1e-9
# Curvature: the kernels take dtheta = atan2(d1 x d2, d1 . d2), the oracle the difference of two atan2 (mlp3:513-536).
# At a nearly collinear joint both are ~1e-16 rad apart in absolute terms, i.e. ~2e-16 / (ds1 + ds2) in kappa; with
# segments >= 1e-6 m (shorter ones give kappa = 0 in both) that is below 1e-9 1/m.
KAP_RTOL, KAP_ATOL = 1e-9, 1e-9
PLAN_SCRATCH_DOUBLES = 320     # fcpp_plan.cu SCRATCH: block-reduction scratch in front of the staged points


@pytest.fixture(scope="module")
def fc():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import field_coverage_path_planning_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def h(fc):
    from field_coverage_path_planning_b200 import _lib
    return _lib.handle(0)


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nan(n):
    import torch
    return torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")


def _nan_summaries(n):
    import torch
    from field_coverage_path_planning_b200 import _lib
    return _nan(max(n, 1) * _lib.SUMMARY_DTYPE.itemsize // 8).view(torch.uint8)


def _summaries(d):
    from field_coverage_path_planning_b200 import _lib
    return d.cpu().numpy().view(_lib.SUMMARY_DTYPE)


# ---------------------------------------------------------------------------------------------------------------
# A. ragged fcpp_speed_verify batches across the length tiers and the HBM-staged kernel
# ---------------------------------------------------------------------------------------------------------------
def _path_caps():
    """cap4, cap2, cap1 (points per path that leave room for 4 / 2 / 1 CTAs per SM, as capacity_for_ctas in
    fcpp_plan.cu computes them: 24 B per point, the reduction scratch and 1 KB per CTA reserved, multiples of 64)
    and the SM count, from the device's properties."""
    import torch
    p = torch.cuda.get_device_properties(0)
    per_sm, optin = p.shared_memory_per_multiprocessor, p.shared_memory_per_block_optin
    fixed = 8 * PLAN_SCRATCH_DOUBLES

    def cap(ctas):
        budget = min(per_sm // ctas - 1024, optin)
        return max(budget - fixed, 0) // 24 // 64 * 64

    return cap(4), cap(2), cap(1), p.multi_processor_count


def _walk(rng, n):
    """A random walk like test_speed_planner_random_paths_vs_oracle's: duplicate points, sharp turns, long jumps."""
    step = rng.normal(0, 1.0, size=(n, 2)) * rng.choice([0.0, 0.3, 1.0, 25.0], size=(n, 1), p=[0.1, 0.3, 0.5, 0.1])
    return np.cumsum(step, axis=0) + rng.uniform(-2000.0, 2000.0, 2), rng.choice([2.5, 4.0, 9.0, 15.0], size=n)


@pytest.fixture(scope="module")
def ragged(fc):
    """~320 paths in shuffled order with lengths on both sides of every tier cap, several longer than the largest
    shared-memory staging (two of them at c and c + stride of path_big_kernel's grid, so that one CTA runs two of
    them), and the oracle's results for each."""
    from oracle import ref_planner as rp
    cap4, cap2, cap1, n_sm = _path_caps()
    assert 256 <= cap4 < cap2 < cap1
    rng = np.random.default_rng(2024)
    n_paths = max(320, 2 * n_sm + 24)
    stride = min(n_paths, 2 * n_sm)                 # path_big_kernel: CTA k takes paths k, k + stride, ...
    big_at = {7: cap1 + 1, 7 + stride: 2 * cap1, stride + 3: cap1 + 2048, n_paths // 2: cap1 + 255}
    assert len(big_at) == 4 and 3 not in big_at
    other = [0, 1, 2, 3, cap4, cap4 + 1, cap2, cap2 + 1, cap1]
    other += list(rng.integers(cap4 - 40, cap2 + 40, size=6))
    other += list(rng.integers(3, 700, size=n_paths - len(big_at) - len(other)))
    other = np.array(other)
    rng.shuffle(other)
    lengths = np.empty(n_paths, dtype=np.int64)
    mask = np.zeros(n_paths, dtype=bool)
    mask[list(big_at)] = True
    lengths[list(big_at)] = list(big_at.values())
    lengths[~mask] = other
    paths, speeds = zip(*(_walk(rng, int(n)) for n in lengths))
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    veh = rp.VehicleParams()
    ref = []
    for p, s in zip(paths, speeds):
        n = len(p)
        planned = rp.speed_plan(p, s, veh)
        kap = np.zeros(n)
        if n >= 3:
            kap[1:-1] = rp.curvatures(p)
        r = dict(n=n, planned=planned, kap=kap, length=rp.path_length(p), t_pre=rp.work_time(p, s),
                 t_post=rp.work_time(p, planned))
        if n >= 3:
            r["cc_planned"] = rp.verify_curvature_constraints(p, planned, veh)
            r["cc_input"] = rp.verify_curvature_constraints(p, s, veh)
        ref.append(r)
    return dict(caps=(cap4, cap2, cap1), n_sm=n_sm, lengths=lengths, offsets=offsets,
                xy=np.ascontiguousarray(np.vstack(paths)), speeds=np.ascontiguousarray(np.concatenate(speeds)), ref=ref)


def _speed_verify(h, batch, max_len, plan=1, alias=False, base=0):
    """One fcpp_speed_verify call on the whole ragged batch, the points placed at ``base`` of NaN-filled buffers.
    Returns (speeds out [base + total + 8], curvature [same], summaries, kernel launches)."""
    import torch
    from field_coverage_path_planning_b200 import VehicleParams, _lib
    v = VehicleParams()
    veh = _lib.Vehicle(v.working_width, v.max_work_speed_kmh, v.max_headland_speed_kmh, v.headland_turn_speed_kmh,
                       v.max_lateral_accel, v.max_longitudinal_accel, v.safety_factor, 2.5)
    total, n_paths = len(batch["speeds"]), len(batch["lengths"])
    size = base + total + 8
    d_xy = _nan(2 * size).view(size, 2)
    d_xy[base:base + total] = torch.from_numpy(batch["xy"]).cuda()
    d_in = _nan(size)
    d_in[base:base + total] = torch.from_numpy(batch["speeds"]).cuda()
    d_off = torch.from_numpy(batch["offsets"] + base).cuda()
    d_out = d_in if alias else _nan(size)
    d_kap = _nan(size)
    d_sum = _nan_summaries(n_paths)
    before = h.launches
    h.check(h.lib.fcpp_speed_verify(h.h, C.byref(veh), d_xy.data_ptr(), d_in.data_ptr(), d_off.data_ptr(), n_paths,
                                    int(max_len), plan, d_out.data_ptr(), d_kap.data_ptr(), d_sum.data_ptr(), _stream()))
    launches = h.launches - before
    return d_out.cpu().numpy(), d_kap.cpu().numpy(), _summaries(d_sum)[:n_paths], launches


def test_speed_verify_ragged_batch_across_tiers_vs_oracle(fc, h, ragged):
    """Speed planning, per-point curvature, length, times and the curvature verification of every path of a batch
    that spans the three shared-memory tiers (256 / 512 / 1024 threads) and the HBM-staged kernel, against
    oracle/ref_planner; then paths of the batch one per call with max_path_len = n, as the drop-in planner calls it
    (a path's thread count depends on its own length only, so the bytes are those of the batch), the same batch
    without speed planning, with the speeds aliased in place, and at a non-zero base offset inside larger buffers."""
    cap4, cap2, cap1 = ragged["caps"]
    lengths, off, ref = ragged["lengths"], ragged["offsets"], ragged["ref"]
    longest = int(lengths.max())
    spd, kap, s, launches = _speed_verify(h, ragged, longest)
    assert launches == 4, launches                  # tiers <= cap4, <= cap2, <= cap1, then the HBM-staged kernel
    print(f"caps: cap4 {cap4} cap2 {cap2} cap1 {cap1}, {len(lengths)} paths, {ragged['n_sm']} SMs, "
          f"{launches} launches")
    worst_v = worst_k = 0.0
    for b, r in enumerate(ref):
        n, o0, o1 = r["n"], int(off[b]), int(off[b + 1])
        rec = s[b]
        assert int(rec["status"]) == 0 and int(rec["n_main"]) == n and int(rec["n_head"]) == 0, (b, n)
        got_v, got_k = spd[o0:o1], kap[o0:o1]
        if n < 3:                                   # mlp3:480-481: fewer than 3 points keep their speeds
            assert got_v.tobytes() == ragged["speeds"][o0:o1].tobytes(), n
        else:
            worst_v = max(worst_v, float(np.abs(got_v - r["planned"]).max()))
            assert np.abs(got_v - r["planned"]).max() <= TIGHT, (b, n)
        if n:
            assert got_k[0] == 0.0 and got_k[-1] == 0.0, (b, n)
            np.testing.assert_allclose(got_k, r["kap"], rtol=KAP_RTOL, atol=KAP_ATOL, err_msg=f"path {b} n={n}")
            worst_k = max(worst_k, float(np.abs(got_k - r["kap"]).max()))
        np.testing.assert_allclose(rec["len_main"], r["length"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(rec["time_main_pre"], r["t_pre"], rtol=1e-9, atol=0)
        np.testing.assert_allclose(rec["time_main"], r["t_post"], rtol=1e-9, atol=0)
        if n >= 3:
            cc = r["cc_planned"]
            assert int(rec["n_accel_viol"]) == cc["accel_violations"], (b, n)
            np.testing.assert_allclose([rec["max_curvature"], rec["max_lateral_accel"], rec["max_jump"]],
                                       [cc["max_curvature"], cc["max_lateral_accel"], cc["max_jump"]],
                                       rtol=1e-9, atol=1e-12, err_msg=f"path {b} n={n}")
        else:
            assert int(rec["n_accel_viol"]) == 0
            assert rec["max_curvature"] == rec["max_lateral_accel"] == rec["max_jump"] == 0.0
    print(f"max |speed - oracle| {worst_v:.3e} km/h, max |kappa - oracle| {worst_k:.3e} 1/m")
    total = int(off[-1])
    assert not np.isnan(spd[:total]).any() and not np.isnan(kap[:total]).any()

    # one path per call, max_path_len = n: the same bytes as inside the batch, on both sides of cap4, cap2 and cap1
    picks = [int(np.flatnonzero((lengths >= 3) & (lengths < cap4))[0])]
    picks += [int(np.flatnonzero(lengths == n)[0]) for n in (cap4, cap4 + 1, cap2, cap2 + 1, cap1, cap1 + 1, 2 * cap1)]
    for b in picks:
        o0, o1 = int(off[b]), int(off[b + 1])
        n = o1 - o0
        one = dict(lengths=lengths[b:b + 1], offsets=np.array([0, n], dtype=np.int64), xy=ragged["xy"][o0:o1],
                   speeds=ragged["speeds"][o0:o1])
        spd1, kap1, s1, _ = _speed_verify(h, one, n)
        assert spd1[:n].tobytes() == spd[o0:o1].tobytes() and kap1[:n].tobytes() == kap[o0:o1].tobytes(), (b, n)
        assert s1.tobytes() == s[b:b + 1].tobytes(), (b, n)

    # verification only: speeds pass through, the counts and maxima are those of the input speeds
    spd0, kap0, s0, _ = _speed_verify(h, ragged, longest, plan=0)
    assert spd0[:total].tobytes() == ragged["speeds"].tobytes()
    assert kap0.tobytes() == kap.tobytes()
    for b, r in enumerate(ref):
        rec = s0[b]
        assert rec["len_main"] == s[b]["len_main"] and rec["time_main_pre"] == s[b]["time_main_pre"]
        np.testing.assert_allclose(rec["time_main"], r["t_pre"], rtol=1e-9, atol=0)
        if r["n"] >= 3:
            cc = r["cc_input"]
            assert int(rec["n_accel_viol"]) == cc["accel_violations"], b
            np.testing.assert_allclose([rec["max_curvature"], rec["max_lateral_accel"], rec["max_jump"]],
                                       [cc["max_curvature"], cc["max_lateral_accel"], cc["max_jump"]],
                                       rtol=1e-9, atol=1e-12, err_msg=f"path {b}")

    # d_speeds_out == d_speeds_in (documented in fcpp.h): byte-identical speeds and summaries
    spd_a, kap_a, s_a, _ = _speed_verify(h, ragged, longest, alias=True)
    assert spd_a.tobytes() == spd.tobytes() and kap_a.tobytes() == kap.tobytes()
    assert s_a.tobytes() == s.tobytes()

    # offsets[0] != 0: the batch inside a larger buffer; nothing outside its points is written
    base = 777
    spd_b, kap_b, s_b, _ = _speed_verify(h, ragged, longest, base=base)
    assert spd_b[base:base + total].tobytes() == spd[:total].tobytes()
    assert kap_b[base:base + total].tobytes() == kap[:total].tobytes()
    assert np.isnan(spd_b[:base]).all() and np.isnan(kap_b[:base]).all()
    assert np.isnan(spd_b[base + total:]).all() and np.isnan(kap_b[base + total:]).all()
    assert s_b.tobytes() == s.tobytes()


@pytest.mark.parametrize("which", ["zero", "below_cap2", "between_cap1_and_longest"])
def test_speed_verify_max_path_len_below_longest_path(fc, h, ragged, which):
    """max_path_len sizes the staging: paths longer than it rounded up to 256 points (max_path_len = 0: longer than
    the largest shared-memory staging, cap1) get FCPP_CAND_TOO_LARGE, a zeroed summary and no speeds or curvature;
    every other path gives exactly what the full-size launch gives."""
    from field_coverage_path_planning_b200 import _lib
    cap4, cap2, cap1 = ragged["caps"]
    lengths, off = ragged["lengths"], ragged["offsets"]
    max_len = {"zero": 0, "below_cap2": cap4 + 700, "between_cap1_and_longest": cap1 + 1000}[which]
    capacity = -(-max_len // 256) * 256 if max_len > 0 else cap1
    assert 0 < (lengths > capacity).sum() < len(lengths)
    spd, kap, s, _ = _speed_verify(h, ragged, int(lengths.max()))
    spd_c, kap_c, s_c, _ = _speed_verify(h, ragged, max_len)
    for b, n in enumerate(lengths):
        o0, o1 = int(off[b]), int(off[b + 1])
        rec = s_c[b]
        if n > capacity:
            assert int(rec["status"]) == _lib.CAND_TOO_LARGE and int(rec["n_main"]) == n, (b, n)
            assert int(rec["n_head"]) == 0 and int(rec["n_accel_viol"]) == 0
            for k in ("len_main", "time_main", "time_main_pre", "max_curvature", "max_lateral_accel", "max_jump"):
                assert rec[k] == 0.0, (b, k)
            assert np.isnan(spd_c[o0:o1]).all() and np.isnan(kap_c[o0:o1]).all(), (b, n)
        else:
            assert rec.tobytes() == s[b].tobytes(), (b, n)
            assert spd_c[o0:o1].tobytes() == spd[o0:o1].tobytes() and kap_c[o0:o1].tobytes() == kap[o0:o1].tobytes()


# ---------------------------------------------------------------------------------------------------------------
# B / C. generated plans: per-point curvature, offsets beyond one scan tile
# ---------------------------------------------------------------------------------------------------------------
def _plan_paths(fc, fields, cand, want_curvature, obstacles=None, coverage=True, **kw):
    """plan_batch(..., outputs='paths') into NaN-filled output buffers.  Returns (BatchResult, the total number of
    points the layout pass reported)."""
    import torch
    from field_coverage_path_planning_b200 import _lib, batch as B
    dev = torch.device("cuda", 0)
    h = _lib.handle(0)
    pb = B.prepare_batch(fields, fc.VehicleParams(), cand, obstacles, None, 0.1, coverage, **kw)
    db = B.DeviceBatch(pb, dev)
    d_off = torch.empty(pb.n_cand + 1, dtype=torch.int64, device=dev)
    h.check(h.lib.fcpp_layout(h.h, C.byref(db.c), None, d_off.data_ptr(), _stream()))
    total = int(h.lib.fcpp_last_total_points(h.h))
    assert total > 0
    buf = B.BatchBuffers(dev, pb.n_cand, pb.n_fields, total, want_curvature)
    for t in (buf.d_path, buf.d_spd, buf.d_kap, buf.d_sum.view(torch.float64)):
        if t is not None:
            t.fill_(float("nan"))
    return B.run_device_batch(db, "paths", want_curvature, buffers=buf), total


def _oracle(fields, cand, b, obstacles=None, **kw):
    from oracle import batch as ob, ref_planner as rp
    return ob.evaluate_candidate(fields[int(cand["field_id"][b])], rp.VehicleParams(),
                                 R=cand["R"][b] if "R" in cand else None,
                                 heading=float(cand["heading"][b]) if "heading" in cand else None,
                                 start_corner=int(cand["start_corner"][b]) if "start_corner" in cand else None,
                                 obstacles=obstacles or (), coverage=False, keep_paths=True, **kw)


def test_plan_curvature_output_vs_oracle(fc):
    """fcpp_outputs.curvature of generated plans at every point — generic points, the regular chains (written from
    the per-candidate table, not from their coordinates), the Ω chains, the main / headland join and both ends —
    against rp.curvatures of the oracle's concatenated plan (the plan is validated as one path).  Asking for the
    curvature changes none of the other outputs."""
    import torch
    from oracle import ref_planner as rp
    cases = [
        ([RECT], fc.make_candidates(1, radii=[5.0, 7.2, 9.6, 12.0], start_corners=[0, 1, 2, 3]), dict(obstacles=[OBST2])),
        ([PARA], fc.make_candidates(1, headings=np.deg2rad([0.0, 17.0, 90.0, 133.0]), radii=[6.0, 9.0]), {}),
        ([RECT, PARA, SMALL], fc.make_candidates(3, radii=[5.0, 11.0], start_corners=[0, 2]), dict(turn_model="omega")),
        ([RECT, PARA], fc.make_candidates(2, radii=[6.0, 8.0], start_corners=[0, 3]), dict(turn_model="clothoid")),
    ]
    worst = 0.0
    for fields, cand, kw in cases:
        res, total = _plan_paths(fc, fields, cand, True, **kw)
        plain, _ = _plan_paths(fc, fields, cand, False, **kw)
        assert res.summary.tobytes() == plain.summary.tobytes()
        assert np.array_equal(res.offsets, plain.offsets) and int(res.offsets[-1]) == total
        assert torch.equal(res.d_path[:total], plain.d_path[:total]) and torch.equal(res.d_speeds[:total], plain.d_speeds[:total])
        assert plain.d_curvature is None
        kap_all = res.d_curvature[:total].cpu().numpy()
        assert not np.isnan(kap_all).any()
        okw = {k: v for k, v in kw.items() if k == "turn_model"}
        compared = 0
        for b in range(len(res.summary)):
            o = _oracle(fields, cand, b, kw.get("obstacles", [None])[0], **okw)
            assert int(res.summary["status"][b]) == o["status"], b
            if o["status"]:
                continue
            compared += 1
            o0, o1 = int(res.offsets[b]), int(res.offsets[b + 1])
            p = res.d_path[o0:o1].cpu().numpy()
            assert p.shape == o["path"].shape and np.abs(p - o["path"]).max() <= TIGHT
            got = kap_all[o0:o1]
            want = np.zeros(len(got))
            want[1:-1] = rp.curvatures(o["path"])
            assert got[0] == 0.0 and got[-1] == 0.0
            nm = int(res.summary["n_main"][b])
            np.testing.assert_allclose(got[nm - 2:nm + 2], want[nm - 2:nm + 2], rtol=KAP_RTOL, atol=KAP_ATOL,
                                       err_msg=f"main / headland join, candidate {b} {kw}")
            np.testing.assert_allclose(got, want, rtol=KAP_RTOL, atol=KAP_ATOL, err_msg=f"candidate {b} {kw}")
            worst = max(worst, float(np.abs(got - want).max()))
        assert compared >= len(res.summary) - 2, (compared, kw)
    print(f"max |kappa - oracle| over the generated plans {worst:.3e} 1/m")


@pytest.mark.parametrize("n_cand", [4096, 4097, 12289])
def test_path_offsets_prefix_sum_beyond_one_scan_tile(fc, n_cand):
    """The offsets of a paths-mode batch are a tiled prefix sum (4096 candidates per tile, then a scan of the tile
    sums and an add pass): offsets equal [0] + cumsum(n_main + n_head), the last one the layout's total, and the
    candidates on both sides of each tile boundary are planned where their offsets say."""
    import torch
    rng = np.random.default_rng(n_cand)
    cand = {"field_id": np.zeros(n_cand, dtype=np.int32), "R": rng.uniform(5.0, 8.0, n_cand),
            "start_corner": rng.integers(0, 4, n_cand).astype(np.int32)}
    res, total = _plan_paths(fc, [SMALL], cand, False, coverage=False)
    s = res.summary
    assert (s["status"] == 0).all()
    n = (s["n_main"] + s["n_head"]).astype(np.int64)
    assert len(np.unique(n)) > 3                                   # plans of different lengths
    assert np.array_equal(res.offsets, np.concatenate([[0], np.cumsum(n)]))
    assert int(res.offsets[-1]) == total
    assert not torch.isnan(res.d_path[:total]).any() and not torch.isnan(res.d_speeds[:total]).any()
    for b in sorted({4095, 4096, 8191, 8192, n_cand - 1}):
        if b >= n_cand:
            continue
        o = _oracle([SMALL], cand, b)
        p, v, _ = res.path(b)
        assert p.shape == o["path"].shape, b
        assert np.abs(p - o["path"]).max() <= TIGHT and np.abs(v - o["speeds"]).max() <= TIGHT, b


# ---------------------------------------------------------------------------------------------------------------
# D. per-field argmin on both sides of its kernel switch (16384 candidates / fields)
# ---------------------------------------------------------------------------------------------------------------
def _argmin_rule(status, cost, field, n_fields, base):
    """Lowest cost among status-0 candidates, ties to the lowest index; +inf / -1 for a field without one."""
    best_c = np.full(n_fields, np.inf)
    best_i = np.full(n_fields, -1, dtype=np.int64)
    ok = np.nonzero(status == 0)[0]
    if len(ok):
        order = ok[np.lexsort((ok, cost[ok], field[ok]))]
        f = field[order]
        first = order[np.concatenate([[True], f[1:] != f[:-1]])]
        best_c[field[first]] = cost[first]
        best_i[field[first]] = first + base
    return best_c, best_i


def _device_argmin(h, sm, cand_field, n_fields, kind, base):
    import torch
    from field_coverage_path_planning_b200 import _lib
    d_sum = torch.from_numpy(np.ascontiguousarray(sm).view(np.uint8).reshape(-1) if len(sm) else
                             np.zeros(_lib.SUMMARY_DTYPE.itemsize, dtype=np.uint8)).cuda()
    d_cf = torch.from_numpy(np.ascontiguousarray(cand_field, dtype=np.int32) if len(sm) else
                            np.zeros(1, dtype=np.int32)).cuda()
    d_cost = _nan(max(n_fields, 1))
    d_best = _nan(max(n_fields, 1)).view(torch.int64)
    h.check(h.lib.fcpp_field_argmin(h.h, d_sum.data_ptr(), d_cf.data_ptr(), len(sm), n_fields, kind, base,
                                    d_cost.data_ptr(), d_best.data_ptr(), _stream()))
    return d_cost.cpu().numpy()[:n_fields], d_best.cpu().numpy()[:n_fields]


def _argmin_summaries(rng, n):
    from field_coverage_path_planning_b200 import _lib
    sm = np.zeros(n, dtype=_lib.SUMMARY_DTYPE)
    # quarter-metre / half-second steps: the sums are exact and ties are common
    sm["len_main"] = rng.integers(0, 40, n) * 0.25
    sm["len_head"] = rng.integers(0, 8, n) * 0.5
    sm["time_main"] = rng.integers(0, 30, n) * 0.5
    sm["time_head"] = rng.integers(0, 6, n) * 1.0
    sm["status"] = np.where(rng.random(n) < 0.2, rng.choice([1, 2, 8, 16], n), 0)
    return sm


@pytest.mark.parametrize("n_fields", [1, 7, 16384, 16385])
@pytest.mark.parametrize("n_cand", [0, 1, 33, 16384, 16385, 200003])
def test_field_argmin_both_kernels_vs_numpy_rule(fc, h, n_cand, n_fields):
    """Explicit cand_field in random order (nearly every warp holds several fields), quantised costs (exact ties
    across warps), dead candidates, both cost kinds, candidate bases 0 and 3 * 2^32."""
    rng = np.random.default_rng(n_cand * 31 + n_fields)
    sm = _argmin_summaries(rng, n_cand)
    field = rng.integers(0, n_fields, n_cand).astype(np.int32)
    for kind in (0, 1):
        cost = sm["len_main"] + sm["len_head"] if kind == 0 else sm["time_main"] + sm["time_head"]
        for base in (0, 3 << 32):
            got_c, got_i = _device_argmin(h, sm, field, n_fields, kind, base)
            want_c, want_i = _argmin_rule(sm["status"], cost, field, n_fields, base)
            assert np.array_equal(got_i, want_i), (kind, base, np.nonzero(got_i != want_i)[0][:5])
            assert np.array_equal(got_c, want_c), (kind, base)


def test_field_argmin_switch_does_not_change_the_answer(fc, h):
    """One dead candidate more (16384 -> 16385 candidates) or one empty field more (16384 -> 16385 fields) moves the
    argmin from the one-CTA kernel to the four-kernel path; the answer is the same bytes."""
    rng = np.random.default_rng(77)
    n = 16384
    sm = _argmin_summaries(rng, n)
    field = rng.integers(0, 512, n).astype(np.int32)
    a_c, a_i = _device_argmin(h, sm, field, 512, 0, 0)
    dead = np.concatenate([sm, sm[:1]])
    dead["status"][-1] = 1
    dead["len_main"][-1] = -1.0                 # would win every field if it were counted
    b_c, b_i = _device_argmin(h, dead, np.concatenate([field, [0]]), 512, 0, 0)
    assert a_c.tobytes() == b_c.tobytes() and a_i.tobytes() == b_i.tobytes()
    field = rng.integers(0, n, n).astype(np.int32)
    a_c, a_i = _device_argmin(h, sm, field, n, 1, 5)
    b_c, b_i = _device_argmin(h, sm, field, n + 1, 1, 5)
    assert a_c.tobytes() == b_c[:n].tobytes() and a_i.tobytes() == b_i[:n].tobytes()
    assert np.isinf(b_c[n]) and b_i[n] == -1


def test_plan_batch_shuffled_field_order_argmin(fc):
    """plan_batch accepts explicit candidates in any field order: its argmin equals NumPy's over its own summary."""
    rng = np.random.default_rng(5)
    fields = [RECT, PARA, SMALL, DEAD, [(0, 0), (120, 0), (120, 90), (0, 90)]]
    cand = fc.make_candidates(len(fields), radii=[5.0, 6.0, 7.5, 8.0, 9.0, 11.0], start_corners=[0, 1, 2, 3])
    perm = rng.permutation(len(cand["field_id"]))
    cand = {k: v[perm] for k, v in cand.items()}
    for cost in ("length", "time"):
        res = fc.plan_batch(fields, fc.VehicleParams(), cand, coverage=False, cost=cost)
        s = res.summary
        c = s["len_main"] + s["len_head"] if cost == "length" else s["time_main"] + s["time_head"]
        want_c, want_i = _argmin_rule(s["status"], c, cand["field_id"], len(fields), 0)
        assert np.array_equal(res.best_cand, want_i) and np.array_equal(res.best_cost, want_c), cost
        assert want_i[3] == -1 and (want_i[[0, 1, 2, 4]] >= 0).all()


# ---------------------------------------------------------------------------------------------------------------
# F. window raster with several row tiles and point chunks
# ---------------------------------------------------------------------------------------------------------------
def _crossing_polyline(rng, n, ox, oy, size, inside):
    """n points on a circle well outside the window [ox, ox + size]^2, except the indices in ``inside``, which are
    uniform in the window: only the segments next to those points reach it."""
    cx, cy = ox + size / 2, oy + size / 2
    th = np.cumsum(rng.normal(0, 0.002, n)) + rng.uniform(0, 2 * np.pi)
    p = np.stack([cx + 1.5 * size * np.cos(th), cy + 1.5 * size * np.sin(th)], axis=1)
    idx = np.array(sorted(k for k in inside if k < n))
    p[idx] = np.stack([ox + rng.uniform(0, size, len(idx)), oy + rng.uniform(0, size, len(idx))], axis=1)
    return p


@pytest.mark.parametrize("R,g", [(25.62, 512), (25.67, 513), (30.02, 600), (60.02, 1200)])
def test_raster_window_row_tiles_and_point_chunks_vs_oracle(fc, R, g):
    """window_kernel keeps min(1024, 8192 / ceil(g / 32)) rows per tile (g = 512: one tile, 513 and 600: two,
    1200: six) and reads the polyline in 1024-point chunks that overlap by one point.  Polylines of 1023 ... ~3000
    points cross the window with the segments around the chunk boundaries; grid and both counts bit for bit against
    the integer oracle."""
    from oracle import raster
    assert int(2 * R / 0.1) == g
    pl = fc.TwoLayerPathPlannerV37(fc.VehicleParams(min_turn_radius=R), field_length=500, field_width=200)
    W = 3.2
    rng = np.random.default_rng(g)
    near_chunks = {1022, 1023, 1024, 1025, 2045, 2046, 2047, 2048}   # chunks start at points 0, 1023, 2046
    for trial, (n1, n2) in enumerate(((1023, 1024), (1025, 2047), (2048, 3001))):
        ci = (trial + g) % 4
        corner = (float(rng.uniform(50, 400)), float(rng.uniform(50, 150)))
        ox = corner[0] if ci in (0, 3) else corner[0] - 2 * R
        oy = corner[1] if ci in (0, 1) else corner[1] - 2 * R
        extra = set(rng.integers(0, 3000, 3).tolist())
        turn = _crossing_polyline(rng, n1, ox, oy, 2 * R, near_chunks | extra)
        rev = _crossing_polyline(rng, n2, ox, oy, 2 * R, near_chunks | extra)
        if n2 > 2047:
            rev[2047] = rev[2046]                                   # a zero-length segment at a chunk boundary
        got = pl.verify_corner_coverage_grid_based(corner, ci, turn, rev)
        c1, bits = raster.raster_window(turn, W / 2, (ox, oy), 0.1, g, g)
        c2, bits = raster.raster_window(rev, W / 2, (ox, oy), 0.1, g, g, bits)
        want = np.unpackbits(bits, bitorder="little")[:g * g].reshape(g, g).astype(bool)
        assert got["grid"].shape == (g, g)
        assert (got["cells_before"], got["cells_after"]) == (c1, c2), (trial, n1, n2)
        assert np.array_equal(got["grid"], want), (trial, n1, n2)
        assert 0 < c1 < c2 < g * g                                  # not saturated: every segment can be missed
