"""numpy statement of the per-field top-k selection (include/fcpp.h, fcpp_selection; DESIGN.md §3.8).

Test infrastructure only: the package never imports it.  ``sel`` is any object with the attributes of
``field_coverage_path_planning_b200.Selection`` (weights, limits as None or int, ``min_coverage`` None or float,
``top_k``).  Every FP64 operation is the library's, in the same order, so costs compare bit for bit.
"""
from __future__ import annotations

import numpy as np


def cost(summary: np.ndarray, sel, cell_area: float) -> np.ndarray:
    """[B] float64: w_length*L + w_time*T + w_boundary*nb + w_obstacle*no + w_accel*na + w_uncovered*U, left to right."""
    s = summary
    L = s["len_main"] + s["len_head"]
    T = s["time_main"] + s["time_head"]
    U = (s["cov_total"] - s["cov_cells"]).astype(np.float64) * np.float64(cell_area)
    c = np.float64(sel.w_length) * L
    c = c + np.float64(sel.w_time) * T
    c = c + np.float64(sel.w_boundary) * s["n_boundary_viol"].astype(np.float64)
    c = c + np.float64(sel.w_obstacle) * s["n_obstacle_viol"].astype(np.float64)
    c = c + np.float64(sel.w_accel) * s["n_accel_viol"].astype(np.float64)
    c = c + np.float64(sel.w_uncovered) * U
    return c


def eligible(summary: np.ndarray, sel) -> np.ndarray:
    """[B] bool: status 0, every set limit held, and the coverage share when min_coverage is set (FP64)."""
    s = summary
    ok = s["status"] == 0
    for name, col in (("max_boundary_viol", "n_boundary_viol"), ("max_obstacle_viol", "n_obstacle_viol"),
                      ("max_accel_viol", "n_accel_viol")):
        lim = getattr(sel, name)
        if lim is not None:
            ok &= s[col] <= int(lim)
    if sel.min_coverage is not None:
        ok &= (s["cov_total"] > 0) & (s["cov_cells"].astype(np.float64) >=
                                      np.float64(sel.min_coverage) * s["cov_total"].astype(np.float64))
    return ok


def rank(summary: np.ndarray, cand_field: np.ndarray, n_fields: int, sel, cell_area: float, base: int = 0):
    """-> (cost [F, k] float64, cand [F, k] int64): per field the eligible candidates ordered by (cost, base + index),
    the first k; +inf / -1 where there are fewer."""
    k = int(sel.top_k)
    out_c = np.full((n_fields, k), np.inf)
    out_i = np.full((n_fields, k), -1, dtype=np.int64)
    fid = np.asarray(cand_field, dtype=np.int64)
    ok = eligible(summary, sel) & (fid >= 0) & (fid < n_fields)
    idx = np.nonzero(ok)[0]
    if len(idx) == 0:
        return out_c, out_i
    c = cost(summary[idx], sel, cell_area)
    f = fid[idx]
    g = idx.astype(np.int64) + int(base)
    # order_bits(cost) as the sort key of the cost: the same total order as the device keys (-0 < +0)
    b = c.view(np.uint64)
    key = np.where(b >> np.uint64(63) == 1, ~b, b | np.uint64(1 << 63))
    o = np.lexsort((g, key, f))
    f, c, g = f[o], c[o], g[o]
    start = np.searchsorted(f, np.arange(n_fields), side="left")
    pos = np.arange(len(f)) - start[f]
    keep = pos < k
    out_c[f[keep], pos[keep]] = c[keep]
    out_i[f[keep], pos[keep]] = g[keep]
    return out_c, out_i


def merge(costs, cands, k: int):
    """The union of the ranks' rankings ([F, k] each), re-ranked by (cost, index): what fcpp_field_select_merge
    computes."""
    c = np.concatenate(costs, axis=1)
    i = np.concatenate(cands, axis=1)
    F = c.shape[0]
    out_c = np.full((F, k), np.inf)
    out_i = np.full((F, k), -1, dtype=np.int64)
    for f in range(F):
        real = i[f] >= 0
        b = c[f][real].view(np.uint64)
        key = np.where(b >> np.uint64(63) == 1, ~b, b | np.uint64(1 << 63))
        o = np.lexsort((i[f][real], key))[:k]
        out_c[f, :len(o)] = c[f][real][o]
        out_i[f, :len(o)] = i[f][real][o]
    return out_c, out_i


def adversarial_summaries(seed: int, n_cand: int, n_fields: int, shuffle: bool = True):
    """Synthetic summaries that stress the ranking: exact cost ties (lengths from a few values), violation counts
    around small limits, coverage at and around the thresholds of ``adversarial_selections``, failed statuses and
    fields without any eligible candidate (the last field of every 7 has only failed ones).  -> (summary [B],
    cand_field [B] int32, field-major unless ``shuffle``)."""
    from field_coverage_path_planning_b200 import _lib
    rng = np.random.default_rng(seed)
    B = int(n_cand)
    s = np.zeros(B, dtype=_lib.SUMMARY_DTYPE)
    fid = np.sort(rng.integers(0, max(n_fields, 1), size=B)).astype(np.int32) if n_fields else np.zeros(0, np.int32)
    s["status"] = np.where(rng.random(B) < 0.1, rng.choice([1, 2, 8, 16], size=B), 0)
    s["status"][(fid % 7) == 6] = 2
    s["len_main"] = rng.choice([100.0, 100.5, 250.25, 1e3 / 3], size=B)
    s["len_head"] = rng.choice([0.0, 50.0, 0.1], size=B)
    s["time_main"] = rng.choice([10.0, 20.0, 7.5], size=B)
    s["time_head"] = rng.choice([0.0, 3.0], size=B)
    for col in ("n_boundary_viol", "n_obstacle_viol", "n_accel_viol"):
        s[col] = rng.integers(0, 5, size=B)
    tot = rng.choice([0, 1000, 1000, 4096, 3], size=B).astype(np.int64)
    # cells exactly at 0.75 and at 0.9 of the total, one below, one above, or anything
    pick = rng.integers(0, 5, size=B)
    cells = np.select([pick == 0, pick == 1, pick == 2, pick == 3],
                      [np.floor(0.75 * tot), np.floor(0.9 * tot), np.floor(0.75 * tot) - 1, np.ceil(0.9 * tot) + 1],
                      rng.integers(0, 4097, size=B))
    s["cov_total"] = tot
    s["cov_cells"] = np.clip(cells, 0, tot).astype(np.int64)
    if shuffle:
        o = rng.permutation(B)
        s, fid = s[o], fid[o]
    return s, fid


def adversarial_selections():
    """Selections (as plain attribute objects) over the same thresholds as ``adversarial_summaries``."""
    from types import SimpleNamespace as NS

    def sel(**kw):
        d = dict(w_length=1.0, w_time=0.0, w_boundary=0.0, w_obstacle=0.0, w_accel=0.0, w_uncovered=0.0,
                 max_boundary_viol=None, max_obstacle_viol=None, max_accel_viol=None, min_coverage=None, top_k=1)
        d.update(kw)
        return NS(**d)
    return [sel(), sel(w_length=0.0, w_time=1.0, top_k=2),
            sel(max_boundary_viol=2, max_obstacle_viol=0, top_k=7),
            sel(min_coverage=0.75, w_uncovered=0.5, top_k=32),
            sel(min_coverage=0.9, max_accel_viol=3, w_boundary=10.0, w_obstacle=2.5, w_accel=0.125, w_time=1.0,
                top_k=7),
            sel(w_length=0.0, top_k=32),                       # every eligible cost 0: ranked by index alone
            sel(min_coverage=1.0, max_boundary_viol=0, max_obstacle_viol=0, max_accel_viol=0, top_k=2),
            # sel()'s twin with a limit no candidate reaches: the same ranking, but not a plain selection, so the
            # library ranks it with the general pipeline at k = 1 instead of the argmin kernels
            sel(max_accel_viol=2**31 - 1)]
