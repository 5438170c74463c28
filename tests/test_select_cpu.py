"""CPU tests of the per-field top-k selection (plan_batch(select=...)): input validation, the fcpp_selection ctypes
mirror, the numpy statement in oracle/select.py against a brute-force sort, and the CPU/gloo form of the multi-GPU
merge over two processes.  The device kernels are pinned to the same oracle by tests/test_gpu_select.py."""
import ctypes
import os
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECT = [(0, 0), (500, 0), (500, 200), (0, 200)]


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    import field_coverage_path_planning_b200 as fc
    return fc


@pytest.mark.parametrize("kw", [
    dict(w_length=-1.0), dict(w_time=float("nan")), dict(w_boundary=float("inf")), dict(w_obstacle=-1e-300),
    dict(w_accel="1"), dict(w_uncovered=True), dict(top_k=0), dict(top_k=33), dict(top_k=2.0),
    dict(max_boundary_viol=-1), dict(max_obstacle_viol=1.5), dict(max_accel_viol=-3), dict(min_coverage=-0.01),
    dict(min_coverage=1.01), dict(min_coverage=float("nan"))])
def test_selection_rejects_bad_values(kw):
    import field_coverage_path_planning_b200 as fc
    with pytest.raises(ValueError):
        fc.Selection(**kw)


def test_selection_accepts_its_range():
    import field_coverage_path_planning_b200 as fc
    s = fc.Selection(w_length=0, w_time=2, w_uncovered=0.5, max_boundary_viol=0, max_obstacle_viol=3,
                     max_accel_viol=np.int64(1), min_coverage=1, top_k=32)
    c = s.c_struct(0.05)
    assert c.top_k == 32 and c.max_boundary_viol == 0 and c.max_accel_viol == 1 and c.min_coverage == 1.0
    assert c.cell_area == 0.05 * 0.05
    d = fc.Selection().c_struct(0.1)
    assert (d.w_length, d.w_time, d.top_k) == (1.0, 0.0, 1)
    assert d.max_boundary_viol == d.max_obstacle_viol == d.max_accel_viol == -1 and d.min_coverage == -1.0


def test_plan_batch_rejects_bad_selections():
    """Refused before any device work: the combinations have no meaning."""
    import field_coverage_path_planning_b200 as fc
    with pytest.raises(ValueError):
        fc.plan_batch([RECT], select=fc.Selection(), cost="time")
    with pytest.raises(ValueError):
        fc.plan_batch([RECT], select=fc.Selection(min_coverage=0.5), coverage=False)
    with pytest.raises(ValueError):
        fc.plan_batch([RECT], select=fc.Selection(w_uncovered=1.0), coverage=False)
    with pytest.raises(ValueError):
        fc.plan_batch([RECT], select={"top_k": 3})
    with pytest.raises(ValueError):
        fc.plan_batch([RECT], select=fc.Selection(), cost="time", distributed=True)


def test_selection_mirror_matches_c_layout(built, tmp_path):
    """sizeof/offsetof of fcpp_selection (gcc on include/fcpp.h) == the ctypes mirror."""
    from field_coverage_path_planning_b200 import _lib
    names = [n for n, _ in _lib.SelectionC._fields_]
    src = tmp_path / "sel.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fcpp.h"\nint main(){printf("%zu %d",'
                   'sizeof(fcpp_selection),FCPP_SELECT_MAX_K);' +
                   "".join(f'printf(" %zu",offsetof(fcpp_selection,{n}));' for n in names) + 'return 0;}')
    exe = tmp_path / "sel"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)]).split()))
    assert got[0] == ctypes.sizeof(_lib.SelectionC) == 80
    assert got[1] == _lib.SELECT_MAX_K
    assert got[2:] == [getattr(_lib.SelectionC, n).offset for n in names]


def _brute(summary, fid, F, sel, cell_area, base=0):
    """The rule of include/fcpp.h in plain Python, one candidate at a time."""
    k = sel.top_k
    rows = [[] for _ in range(F)]
    for i, s in enumerate(summary):
        if int(s["status"]) != 0:
            continue
        nb, no, na = int(s["n_boundary_viol"]), int(s["n_obstacle_viol"]), int(s["n_accel_viol"])
        if (sel.max_boundary_viol is not None and nb > sel.max_boundary_viol) or \
                (sel.max_obstacle_viol is not None and no > sel.max_obstacle_viol) or \
                (sel.max_accel_viol is not None and na > sel.max_accel_viol):
            continue
        cells, tot = int(s["cov_cells"]), int(s["cov_total"])
        if sel.min_coverage is not None and not (tot > 0 and float(cells) >= sel.min_coverage * float(tot)):
            continue
        L = float(s["len_main"]) + float(s["len_head"])
        T = float(s["time_main"]) + float(s["time_head"])
        U = float(tot - cells) * cell_area
        c = sel.w_length * L + sel.w_time * T + sel.w_boundary * float(nb) + sel.w_obstacle * float(no) + \
            sel.w_accel * float(na) + sel.w_uncovered * U
        rows[int(fid[i])].append((c, base + i))
    cost = np.full((F, k), np.inf)
    cand = np.full((F, k), -1, dtype=np.int64)
    for f, r in enumerate(rows):
        r.sort()
        for j, (c, i) in enumerate(r[:k]):
            cost[f, j], cand[f, j] = c, i
    return cost, cand


@pytest.mark.parametrize("seed,B,F", [(0, 0, 0), (1, 0, 5), (2, 1, 1), (3, 300, 1), (4, 2000, 37), (5, 500, 200)])
def test_oracle_matches_brute_force(built, seed, B, F):
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(seed, B, F)
    for sel in osel.adversarial_selections():
        for cell_area in (0.01, 0.0025):
            want = _brute(summ, fid, F, sel, cell_area, base=17)
            got = osel.rank(summ, fid, F, sel, cell_area, base=17)
            assert np.array_equal(got[1], want[1])
            assert got[0].tobytes() == want[0].tobytes()


def test_adversarial_inputs_hit_the_edges(built):
    """The synthetic inputs do contain what the tests claim: ties, limits at n == max and max + 1, coverage exactly
    at the threshold, fields with no eligible candidate and fields with fewer than k."""
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(4, 2000, 37)
    sels = osel.adversarial_selections()
    c = osel.cost(summ, sels[0], 0.01)
    assert len(np.unique(c)) < len(c) // 10                                 # many exact ties
    nb = summ["n_boundary_viol"]
    assert (nb == 2).any() and (nb == 3).any()
    cov = summ["cov_total"] > 0
    at = summ["cov_cells"][cov].astype(np.float64) == 0.75 * summ["cov_total"][cov].astype(np.float64)
    assert at.any()
    _, cand = osel.rank(summ, fid, 37, sels[3], 0.01)
    assert (cand[:, 0] == -1).any()                                          # all-ineligible fields
    assert ((cand[:, 0] >= 0) & (cand[:, -1] == -1)).any()                   # fewer than k eligible


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir, B, F):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from field_coverage_path_planning_b200 import _lib, dist as fdist
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(11, B, F)
    lo, hi = fdist.shard_range(B, world, rank)
    out = []
    for sel in osel.adversarial_selections():
        k = sel.top_k
        cost, cand = osel.rank(summ[lo:hi], fid[lo:hi], F, sel, 0.01, base=lo)
        t_cost, t_cand = torch.from_numpy(cost.copy()), torch.from_numpy(cand.copy())
        fdist.reduce_topk(t_cost, t_cand, k)
        rec = fdist.gather_winner_records(torch.from_numpy(summ[lo:hi].view(np.uint8).reshape(-1).copy()),
                                          t_cand.reshape(-1), lo, hi)
        out += [t_cost.numpy().reshape(-1), t_cand.numpy().reshape(-1).astype(np.float64),
                rec.numpy().view(_lib.SUMMARY_DTYPE).reshape(-1)["len_main"]]
    np.save(os.path.join(out_dir, f"r{rank}.npy"), np.concatenate(out))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_topk_merge_world2(built, tmp_path):
    """Two gloo ranks rank their halves, merge with dist.reduce_topk and gather the ranked records: every rank holds
    the single-process ranking of the union, and the records of the ranked candidates."""
    from oracle import select as osel
    B, F = 1500, 23
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), B, F), nprocs=world, join=True)
    r0, r1 = np.load(tmp_path / "r0.npy"), np.load(tmp_path / "r1.npy")
    assert r0.tobytes() == r1.tobytes()
    summ, fid = osel.adversarial_summaries(11, B, F)
    at = 0
    for sel in osel.adversarial_selections():
        n = F * sel.top_k
        cost, cand = osel.rank(summ, fid, F, sel, 0.01)
        assert r0[at:at + n].tobytes() == cost.reshape(-1).tobytes()
        assert np.array_equal(r0[at + n:at + 2 * n], cand.reshape(-1).astype(np.float64))
        c = cand.reshape(-1)
        want_len = np.where(c >= 0, summ["len_main"][np.maximum(c, 0)], 0.0)
        assert np.array_equal(r0[at + 2 * n:at + 3 * n], want_len)
        at += 3 * n
    assert at == len(r0)


def test_oracle_merge_equals_ranking_of_the_union(built):
    """oracle.select.merge of per-shard rankings (the device merge's statement) == the ranking of the whole set,
    for uneven shard splits."""
    from field_coverage_path_planning_b200 import dist as fdist
    from oracle import select as osel
    summ, fid = osel.adversarial_summaries(12, 3000, 41)
    for sel in osel.adversarial_selections():
        for world in (2, 3, 8):
            parts = [osel.rank(summ[lo:hi], fid[lo:hi], 41, sel, 0.01, base=lo)
                     for lo, hi in (fdist.shard_range(3000, world, r) for r in range(world))]
            got = osel.merge([p[0] for p in parts], [p[1] for p in parts], sel.top_k)
            want = osel.rank(summ, fid, 41, sel, 0.01)
            assert np.array_equal(got[1], want[1]) and got[0].tobytes() == want[0].tobytes()
