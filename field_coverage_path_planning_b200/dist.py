"""Multi-GPU: one process per GPU (torch.distributed), candidates sharded in contiguous ranges,
NO data-path collective — the only exchange is the final per-field ranking (SURVEY.md §8(e)).

The reduction is exact and deterministic (ties go to the lowest global candidate index):
    1+2. CUDA: ONE all-gather of every rank's [F, k] costs and candidates and the library's merge kernel
       (fcpp_field_select_merge; k = 1 is the per-field argmin).  CPU/gloo (tests): an all-gather and a sort;
    3. the records of the F * k ranked candidates are contributed by their owners (fcpp_winner_records) and summed
       as int32 words (every other rank contributes zeros), i.e. an all-gather of k records per field.
Works on NCCL (CUDA tensors) and gloo (CPU tensors — used by the world_size-2 CPU tests).
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib

I64_MAX = torch.iinfo(torch.int64).max


def shard_range(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced shard [lo, hi) of n candidates for `rank` (first n % world ranks get one more)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_candidates(cands: Dict[str, np.ndarray], world: int, rank: int) -> Tuple[Dict[str, np.ndarray], int]:
    """The rank's contiguous shard of a candidate set + its first global index.  Factored sets
    (batch.candidate_axes) keep their axes and get a ``range`` — nothing is sliced or copied."""
    from .batch import axes_count, is_axes
    if is_axes(cands):
        first = int(cands.get("range", (0, 0))[0])
        lo, hi = shard_range(axes_count(cands), world, rank)
        return dict(cands, range=(first + lo, first + hi)), first + lo
    n = len(cands["field_id"])
    lo, hi = shard_range(n, world, rank)
    return {k: v[lo:hi] for k, v in cands.items()}, lo


def reduce_best(best_cost: torch.Tensor, best_cand: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Global per-field (cost, candidate) [F] from the local ones (``best_cand``: GLOBAL candidate indices, -1 = none),
    in place: ``reduce_topk`` at k = 1."""
    return reduce_topk(best_cost, best_cand, 1, group)


def reduce_topk(top_cost: torch.Tensor, top_cand: torch.Tensor, k: int, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Global per-field top-k from the ranks' local ones, in place.  ``top_cost`` / ``top_cand`` hold [F, k] (flat
    or 2-D) sorted by (cost, GLOBAL candidate index), padded with +inf / -1; the result is the k lowest
    (cost, index) of the union, padded the same way.

    CUDA tensors: one NCCL all-gather of the 2 F k words + the library's merge kernel (fcpp_field_select_merge).
    CPU tensors (gloo tests): the same rule with torch ops."""
    n = top_cost.numel()
    F = n // k if k else 0
    world = dist.get_world_size(group)
    if top_cost.is_cuda:
        import ctypes as C
        dev = top_cost.device
        adjacent = (top_cost.dtype == torch.float64 and top_cand.dtype == torch.int64 and top_cost.is_contiguous()
                    and top_cand.is_contiguous() and top_cand.data_ptr() == top_cost.data_ptr() + 8 * n
                    and top_cost.untyped_storage().data_ptr() == top_cand.untyped_storage().data_ptr())
        if adjacent:   # BatchBuffers lays them out back to back
            send = torch.empty(0, dtype=torch.int64, device=dev).set_(
                top_cost.untyped_storage(), top_cost.storage_offset(), (2 * n,))
        else:
            send = torch.cat([top_cost.reshape(-1).view(torch.int64), top_cand.reshape(-1)])
        gathered = torch.empty(world * 2 * n, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(gathered, send, group=group)
        h = _lib.handle(dev.index)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        h.check(h.lib.fcpp_field_select_merge(h.h, gathered.data_ptr(), world, F, k, top_cost.data_ptr(),
                                              top_cand.data_ptr(), st))
        return top_cost, top_cand
    costs = [torch.empty_like(top_cost) for _ in range(world)]
    cands = [torch.empty_like(top_cand) for _ in range(world)]
    dist.all_gather(costs, top_cost.contiguous(), group=group)
    dist.all_gather(cands, top_cand.contiguous(), group=group)
    c = torch.cat([x.reshape(F, k) for x in costs], dim=1)           # [F, world k]
    i = torch.cat([x.reshape(F, k) for x in cands], dim=1)
    i = torch.where(i < 0, torch.full_like(i, I64_MAX), i)           # padding after every real entry
    c = torch.where(i == I64_MAX, torch.full_like(c, float("inf")), c)
    # (cost, index) order: by index, then STABLY by cost
    o = torch.argsort(i, dim=1, stable=True)
    c, i = torch.gather(c, 1, o), torch.gather(i, 1, o)
    o = torch.argsort(c, dim=1, stable=True)
    c, i = torch.gather(c, 1, o)[:, :k], torch.gather(i, 1, o)[:, :k]
    none = i == I64_MAX
    top_cost.copy_(torch.where(none, torch.full_like(c, float("inf")), c).reshape(top_cost.shape))
    top_cand.copy_(torch.where(none, torch.full_like(i, -1), i).reshape(top_cand.shape))
    return top_cost, top_cand


def gather_winner_records(summary_bytes: torch.Tensor, best_cand: torch.Tensor, lo: int, hi: int,
                          group=None, count_mask: int = 0) -> torch.Tensor:
    """[F, 176] uint8: the summary record of every field's global winner.
    ``summary_bytes`` = this rank's records as a flat uint8 tensor ((hi-lo)*176 bytes).
    CUDA: one library kernel writes the records this rank owns (zeros elsewhere), one all-reduce sums them;
    CPU tensors (gloo tests): the same with torch ops.
    ``count_mask`` != 0 (CUDA): the returned tensor is flat, F * 176 + 16 bytes — behind the records rides one
    int32 word, the number of candidates OF ALL RANKS whose status has a bit of the mask (fcpp_status_count; the
    same all-reduce sums it): every rank learns in the same read-back whether any rank's launch sizes were too
    small, so that all of them repeat the batch together."""
    rec = _lib.SUMMARY_DTYPE.itemsize
    F = best_cand.numel()
    if best_cand.is_cuda:
        import ctypes as C
        dev = best_cand.device
        out = torch.empty(F * rec + (16 if count_mask else 0), dtype=torch.uint8, device=dev)
        h = _lib.handle(dev.index)
        st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        h.check(h.lib.fcpp_winner_records(h.h, summary_bytes.data_ptr() if hi > lo else None, lo, hi,
                                          best_cand.data_ptr(), F, out.data_ptr(), st))
        if count_mask:
            out[F * rec + 4:].zero_()
            h.check(h.lib.fcpp_status_count(h.h, summary_bytes.data_ptr() if hi > lo else None, hi - lo, count_mask,
                                            out.data_ptr() + F * rec, st))
        dist.all_reduce(out.view(torch.int32), op=dist.ReduceOp.SUM, group=group)
        return out if count_mask else out.view(F, rec)
    own = (best_cand >= lo) & (best_cand < hi)
    idx = torch.where(own, best_cand - lo, torch.zeros_like(best_cand))
    rows = summary_bytes.view(-1, rec)[idx] if hi > lo else torch.zeros((F, rec), dtype=torch.uint8,
                                                                        device=best_cand.device)
    rows = torch.where(own[:, None], rows, torch.zeros_like(rows)).contiguous()
    words = rows.view(torch.int32)
    dist.all_reduce(words, op=dist.ReduceOp.SUM, group=group)
    return words.view(torch.uint8).view(F, rec)


def plan_batch_sharded(fields, vehicle, candidates, obstacles, start_points, outputs, grid_h, coverage, cost,
                       device, want_curvature, turn_model="arc", clothoid_share=0.5, winners=False, wait=True,
                       select=None, obstacle_sweep=False):
    """plan_batch over all ranks of the default process group (see batch.plan_batch): every rank plans its
    contiguous shard; ONE all-gather + merge kernel gives every rank the per-field ranking (the argmin of ``cost``, or
    the top-k of ``select``), one kernel + one all-reduce the summary record of every ranked candidate; the local
    summaries, the merged ranking and the records come back to the host with ONE synchronisation.  Launch sizes are
    remembered from earlier batches of the same shape (no layout read-back); ``wait=False`` returns a
    ``batch.PendingBatch``.  With ``obstacle_sweep`` each rank gets the sweep of its own candidates
    (``BatchResult.sweep``)."""
    from .batch import DeviceBatch, _dev, axes_count, is_axes, prepare_batch, run_device_batch
    if not dist.is_initialized():
        raise RuntimeError("distributed=True needs torch.distributed.init_process_group (backend 'nccl')")
    world, rank = dist.get_world_size(), dist.get_rank()
    fv = np.asarray(fields, dtype=np.float64).reshape(-1, 4, 2)
    if candidates is None:
        candidates = {"field_id": np.arange(len(fv), dtype=np.int32)}
    n = axes_count(candidates) if is_axes(candidates) else len(candidates["field_id"])
    local, lo = shard_candidates(candidates, world, rank)
    hi = lo + (axes_count(local) if is_axes(local) else len(local["field_id"]))
    sp = None if start_points is None else np.asarray(start_points, dtype=np.float64).reshape(n, 2)[lo:hi]
    dev = _dev(device)
    pb = prepare_batch(fv, vehicle, local, obstacles, sp, grid_h, coverage, turn_model, clothoid_share)
    db = DeviceBatch(pb, dev)
    return run_device_batch(db, outputs, want_curvature, cost, lo, winners=winners, speculate=True, wait=wait,
                            shard=(lo, hi), select=select, obstacle_sweep=obstacle_sweep)
