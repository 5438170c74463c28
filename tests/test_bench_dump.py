"""bench.py --dump-outputs: what it writes from a step's output buffers (host tensors stand in for the device)."""
import os

import numpy as np
import torch

import bench
from field_coverage_path_planning_b200 import _lib
from field_coverage_path_planning_b200.batch import BatchBuffers


def _buffers(B, F):
    n_pts = np.random.default_rng(0).integers(10, 40, B)
    off = np.concatenate([[0], np.cumsum(n_pts)])
    bufs = BatchBuffers(torch.device("cpu"), B, F, int(off[-1]))
    s = np.zeros(B, dtype=_lib.SUMMARY_DTYPE)
    s["n_main"] = np.arange(B)
    s["cov_total"] = 2 ** 40 + np.arange(B)
    s["corner_after"] = np.arange(4 * B).reshape(B, 4)
    bufs.d_sum.copy_(torch.from_numpy(s.view(np.uint8)))
    bufs.d_off.copy_(torch.from_numpy(off))
    bufs.d_path.copy_(torch.arange(2 * off[-1], dtype=torch.float64).view(-1, 2))
    bufs.d_spd.copy_(torch.arange(off[-1], dtype=torch.float64))
    bufs.d_cost.copy_(torch.tensor([1.5, np.inf, 2.0], dtype=torch.float64))
    bufs.d_best.copy_(torch.tensor([7, -1, 9]))
    return bufs, off


def test_dump_outputs_samples_are_fixed_and_exact(tmp_path, monkeypatch):
    B, F, base = 5000, 3, 100
    bufs, off = _buffers(B, F)
    a = bench.dump_outputs(bufs, B, F, base, True)
    b = bench.dump_outputs(bufs, B, F, base, True)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    assert all(v.dtype == np.float64 for v in a.values())
    assert "summary_reserved" not in a
    np.testing.assert_array_equal(a["best_cost"], [1.5, np.inf, 2.0])
    np.testing.assert_array_equal(a["best_cand"], [7, -1, 9])
    np.testing.assert_array_equal(a["summary_cand"], base + np.arange(B))
    np.testing.assert_array_equal(a["summary_cov_total"], 2 ** 40 + np.arange(B))
    assert a["summary_corner_after"].shape == (B, 4)
    # paths: a seeded sample of DUMP_PATH_ROWS candidates, each one's points in path_offsets order
    pc, po = a["path_cand"].astype(int) - base, a["path_offsets"].astype(int)
    assert len(pc) == bench.DUMP_PATH_ROWS and np.all(np.diff(pc) > 0)
    for i in (0, 17, len(pc) - 1):
        np.testing.assert_array_equal(a["speeds_kmh"][po[i]:po[i + 1]], np.arange(off[pc[i]], off[pc[i] + 1]))
        np.testing.assert_array_equal(a["path_xy"][po[i]:po[i + 1], 0], 2 * np.arange(off[pc[i]], off[pc[i] + 1]))
    bench.write_dump(str(tmp_path / "d"), a)
    assert sorted(os.listdir(tmp_path / "d")) == sorted(k + ".npy" for k in a)
    np.testing.assert_array_equal(np.load(tmp_path / "d" / "path_xy.npy"), a["path_xy"])
    # larger batches: a seeded sample of the summaries, no paths in summary mode
    monkeypatch.setattr(bench, "DUMP_SUMMARY_ROWS", 1000)
    c = bench.dump_outputs(bufs, B, F, 0, False)
    assert len(c["summary_cand"]) == 1000 and "path_xy" not in c
    np.testing.assert_array_equal(c["summary_n_main"], c["summary_cand"])
