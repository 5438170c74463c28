"""Batch entry point: evaluate many candidate plans (fields x heading x turn radius x start
corner) at once on the GPU through libfcpp.so — SURVEY.md §8(b) "New batch entry".

Host side = FP64 numpy set-up of the per-field / per-candidate scalars (A2, mlp3:109-343),
device memory and streams through torch, everything else inside the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field as dc_field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _geometry as G
from . import _lib
from .vehicle import VehicleParams

ROT_THRESHOLD = 0.01  # mlp3:686, :709


def _dev(device) -> torch.device:
    if device is None:
        if not torch.cuda.is_available():
            raise _lib.FcppError("no CUDA device: this package has no CPU path")
        return torch.device("cuda", torch.cuda.current_device())
    d = torch.device(device)
    if d.type != "cuda":
        raise _lib.FcppError(f"device {d} is not a CUDA device: this package has no CPU path")
    if d.index is None:
        d = torch.device("cuda", torch.cuda.current_device())
    return d


class _Staging:
    """Grow-only pinned host buffer of one device and slot: ONE packed host->device copy of a batch's inputs,
    instead of a cudaHostAlloc + copy per array.  (Results are read back into ``_ResultPool`` buffers.)"""
    _per_dev: Dict[tuple, "_Staging"] = {}

    def __init__(self):
        self.h_in = None
        self.in_done = None          # event: the last packed H2D copy has left h_in

    @classmethod
    def get(cls, dev: torch.device, slot: int = 0) -> "_Staging":
        st = cls._per_dev.get((dev.index, slot))
        if st is None:
            st = cls._per_dev[(dev.index, slot)] = cls()
        return st

    def host_in(self, nbytes: int) -> torch.Tensor:
        if self.in_done is not None:
            self.in_done.synchronize()           # the previous copy may still be reading the buffer
        if self.h_in is None or self.h_in.numel() < nbytes:
            self.h_in = torch.empty(max(nbytes * 2, 1 << 20), dtype=torch.uint8).pin_memory()
        return self.h_in


class _PinnedView:
    """numpy's owner object of a view into a pinned buffer: alive exactly as long as some array views it."""

    def __init__(self, t: torch.Tensor, nbytes: int):
        self.t = t
        self.__array_interface__ = {"data": (t.data_ptr(), False), "shape": (int(nbytes),), "typestr": "|u1",
                                    "version": 3}


class _ResultPool:
    """Pinned host buffers that results are read back INTO and handed to the caller as numpy views — no host
    memcpy out of a staging buffer (at 737 280 candidates that copy cost more than the PCIe transfer).  A buffer
    is reused only when no array views it any more (weak reference to the views' owner object), so a caller that
    drops the previous BatchResult runs allocation-free; one that keeps many results gets new buffers up to
    ``MAX_BYTES`` and, beyond that, a pinned buffer per read-back that the pool does not keep.  Every device->host
    read-back takes its host memory from here: no two read-backs that can be in flight share a buffer."""
    MAX_BYTES = 4 << 30
    _bufs: List[list] = []          # [tensor, weakref to the _PinnedView handed out last | None]

    @staticmethod
    def _free(e) -> bool:
        return e[1] is None or e[1]() is None

    @classmethod
    def get(cls, nbytes: int):
        """-> (pinned uint8 tensor, numpy uint8 view of its first nbytes)."""
        import weakref
        nbytes = max(int(nbytes), 256)
        best = None
        for e in cls._bufs:
            if e[0].numel() >= nbytes and cls._free(e) and (best is None or e[0].numel() < best[0].numel()):
                best = e
        if best is None:
            cls._bufs = [e for e in cls._bufs if not cls._free(e)]      # free ones were too small
            if sum(e[0].numel() for e in cls._bufs) + nbytes > cls.MAX_BYTES:
                t = torch.empty(nbytes, dtype=torch.uint8).pin_memory()   # freed with the last view of it
                return t, np.asarray(_PinnedView(t, nbytes))
            best = [torch.empty(max(nbytes + (nbytes >> 2), 1 << 20), dtype=torch.uint8).pin_memory(), None]
            cls._bufs.append(best)
        pv = _PinnedView(best[0], nbytes)
        best[1] = weakref.ref(pv)
        return best[0], np.asarray(pv)


_TORCH_DTYPE = {np.dtype(np.float64).str: torch.float64, np.dtype(np.int32).str: torch.int32,
                np.dtype(np.int64).str: torch.int64, np.dtype(np.uint8).str: torch.uint8}


def _pack_to_dev(arrays: Dict[str, np.ndarray], dev: torch.device, slot: int = 0) -> Dict[str, torch.Tensor]:
    """All input arrays through one pinned staging buffer and one async copy; the device tensors
    are typed views of one allocation (256-byte aligned slices)."""
    offs, total = {}, 0
    for k, a in arrays.items():
        offs[k] = total
        total += (a.nbytes + 255) & ~255
    total = max(total, 256)
    st = _Staging.get(dev, slot)
    h = st.host_in(total)
    hv = h.numpy()
    for k, a in arrays.items():
        hv[offs[k]:offs[k] + a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    with torch.cuda.device(dev):
        d = torch.empty(total, dtype=torch.uint8, device=dev)
        d.copy_(h[:total], non_blocking=True)
        if st.in_done is None:
            st.in_done = torch.cuda.Event()
        st.in_done.record(torch.cuda.current_stream(dev))
    out = {}
    for k, a in arrays.items():
        t = d[offs[k]:offs[k] + a.nbytes].view(_TORCH_DTYPE[a.dtype.str])
        out[k] = t.view(a.shape) if a.nbytes else t
    out["_packed"] = d
    return out


def _to_dev(a: np.ndarray, dev: torch.device, pin: bool = True) -> torch.Tensor:
    t = torch.from_numpy(np.ascontiguousarray(a))
    if pin:
        t = t.pin_memory()
    return t.to(dev, non_blocking=True)


def make_candidates(n_fields: int, headings: Optional[Sequence[float]] = None,
                    radii: Optional[Sequence[float]] = None,
                    start_corners: Optional[Sequence[int]] = None) -> Dict[str, np.ndarray]:
    """Cartesian product field x heading x radius x start corner, field-major (all candidates of
    one field are contiguous).  ``headings`` in radians; ``None`` keeps the reference's heading
    (direction of field edge 0, mlp3:244-263); radii ``None`` keeps the vehicle's radius."""
    hs = [None] if headings is None else list(headings)
    rs = [None] if radii is None else list(radii)
    cs = [None] if start_corners is None else list(start_corners)
    nh, nr, nc = len(hs), len(rs), len(cs)
    per = nh * nr * nc
    B = n_fields * per
    fid = np.repeat(np.arange(n_fields, dtype=np.int32), per)
    idx = np.tile(np.arange(per), n_fields)
    out: Dict[str, np.ndarray] = {"field_id": fid}
    if headings is not None:
        out["heading"] = np.asarray(hs, dtype=np.float64)[idx // (nr * nc)]
    if radii is not None:
        out["R"] = np.asarray(rs, dtype=np.float64)[(idx // nc) % nr]
    if start_corners is not None:
        out["start_corner"] = np.asarray(cs, dtype=np.int32)[idx % nc]
    assert len(fid) == B
    return out


def candidate_axes(n_fields: int, headings: Optional[Sequence[float]] = None,
                   radii: Optional[Sequence[float]] = None,
                   start_corners: Optional[Sequence[int]] = None) -> Dict[str, object]:
    """The same candidate set as ``make_candidates`` (same order, same indices) in FACTORED form: only the
    axes are kept, the library decodes candidate g = ((field * NH + heading) * NR + radius) * NC + corner on
    the device (fcpp_batch: cand_field == NULL).  Nothing per candidate is computed on or copied from the
    host — a 737 280-candidate heading search sends its 180 headings, not 36 MB of candidate arrays."""
    ax: Dict[str, object] = {"axes": True, "n_fields": int(n_fields)}
    if headings is not None:
        ax["heading"] = np.ascontiguousarray(headings, dtype=np.float64).reshape(-1)
    if radii is not None:
        ax["R"] = np.ascontiguousarray(radii, dtype=np.float64).reshape(-1)
    if start_corners is not None:
        ax["start_corner"] = np.ascontiguousarray(start_corners, dtype=np.int32).reshape(-1)
    for k in ("heading", "R", "start_corner"):
        if k in ax and len(ax[k]) == 0:
            raise ValueError(f"empty candidate axis {k!r}")
    return ax


def is_axes(candidates) -> bool:
    return isinstance(candidates, dict) and bool(candidates.get("axes", False))


def axes_per_field(ax) -> int:
    return (len(ax["heading"]) if "heading" in ax else 1) * (len(ax["R"]) if "R" in ax else 1) * \
        (len(ax["start_corner"]) if "start_corner" in ax else 1)


def axes_count(ax) -> int:
    """Number of candidates of a factored set (or of its ``range``)."""
    if "range" in ax:
        return int(ax["range"][1] - ax["range"][0])
    return int(ax["n_fields"]) * axes_per_field(ax)


def expand_axes(ax, index: Optional[np.ndarray] = None) -> Dict[str, np.ndarray]:
    """Explicit candidate arrays (the ``make_candidates`` form) of a factored set, or of the product indices
    ``index`` only (the winners of a search)."""
    nh = len(ax["heading"]) if "heading" in ax else 1
    nr = len(ax["R"]) if "R" in ax else 1
    nc = len(ax["start_corner"]) if "start_corner" in ax else 1
    per = nh * nr * nc
    if index is None:
        lo, hi = ax.get("range", (0, int(ax["n_fields"]) * per))
        index = np.arange(lo, hi, dtype=np.int64)
    g = np.asarray(index, dtype=np.int64)
    rem = g % per
    out: Dict[str, np.ndarray] = {"field_id": (g // per).astype(np.int32)}
    if "heading" in ax:
        out["heading"] = ax["heading"][rem // (nr * nc)]
    if "R" in ax:
        out["R"] = ax["R"][(rem // nc) % nr]
    if "start_corner" in ax:
        out["start_corner"] = ax["start_corner"][rem % nc]
    return out


@dataclass(frozen=True)
class Selection:
    """How ``plan_batch(..., select=...)`` ranks the candidates of each field (include/fcpp.h, fcpp_selection).

    A candidate is eligible when its status is 0, every limit that is set holds (``n_*_viol <= max_*``) and, with
    ``min_coverage`` set, its headland band has cells and ``cov_cells >= min_coverage * cov_total`` (FP64).  Its cost,
    in FP64, left to right::

        w_length * (len_main + len_head) + w_time * (time_main + time_head) + w_boundary * n_boundary_viol
        + w_obstacle * n_obstacle_viol + w_accel * n_accel_viol + w_uncovered * (cov_total - cov_cells) * grid_h**2

    Per field the eligible candidates are ranked by (cost, candidate index) and the first ``top_k`` are returned.
    The defaults are ``cost='length'``'s argmin exactly: same winner, same cost bits."""
    w_length: float = 1.0
    w_time: float = 0.0
    w_boundary: float = 0.0
    w_obstacle: float = 0.0
    w_accel: float = 0.0
    w_uncovered: float = 0.0          # per m² of the headland band left uncovered
    max_boundary_viol: Optional[int] = None
    max_obstacle_viol: Optional[int] = None
    max_accel_viol: Optional[int] = None
    min_coverage: Optional[float] = None    # share of the headland band's cells, in [0, 1]
    top_k: int = 1

    WEIGHTS = ("w_length", "w_time", "w_boundary", "w_obstacle", "w_accel", "w_uncovered")
    LIMITS = ("max_boundary_viol", "max_obstacle_viol", "max_accel_viol")

    def __post_init__(self):
        for n in self.WEIGHTS:
            w = getattr(self, n)
            if isinstance(w, bool) or not isinstance(w, (int, float, np.floating, np.integer)) or \
                    not math.isfinite(float(w)) or float(w) < 0:
                raise ValueError(f"Selection.{n} must be a finite number >= 0, not {w!r}")
        k = self.top_k
        if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= _lib.SELECT_MAX_K:
            raise ValueError(f"Selection.top_k must be an integer in 1..{_lib.SELECT_MAX_K}, not {k!r}")
        for n in self.LIMITS:
            v = getattr(self, n)
            if v is not None and (isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not 0 <= int(v) < 2**31):
                raise ValueError(f"Selection.{n} must be None or an integer >= 0, not {v!r}")
        c = self.min_coverage
        if c is not None and (isinstance(c, bool) or not isinstance(c, (int, float, np.floating, np.integer)) or
                              not 0.0 <= float(c) <= 1.0):
            raise ValueError(f"Selection.min_coverage must be None or in [0, 1], not {c!r}")

    def check_batch(self, coverage: bool, cost: str):
        """The combinations ``plan_batch`` refuses."""
        if cost != "length":
            raise ValueError("select= replaces cost=: weight the time with Selection(w_length=0, w_time=1)")
        if not coverage and (self.min_coverage is not None or self.w_uncovered > 0):
            raise ValueError("min_coverage and w_uncovered need coverage=True: without it the coverage counts are 0, "
                             "not measured")

    def c_struct(self, grid_h: float) -> "_lib.SelectionC":
        def lim(v):
            return -1 if v is None else int(v)
        return _lib.SelectionC(*[float(getattr(self, n)) for n in self.WEIGHTS], float(grid_h) * float(grid_h),
                               -1.0 if self.min_coverage is None else float(self.min_coverage),
                               lim(self.max_boundary_viol), lim(self.max_obstacle_viol), lim(self.max_accel_viol),
                               int(self.top_k))


@dataclass
class PreparedBatch:
    """Host (numpy) side of one batch, ready to be copied to a device."""
    vehicle: VehicleParams
    n_fields: int
    n_cand: int
    arrays: Dict[str, np.ndarray]
    max_obs_verts: int
    max_obs_polys: int
    grid_h: float
    coverage: bool
    turn_model: str = "arc"
    clothoid_share: float = 0.5
    dedupe: int = 0          # fcpp_batch.cover_dedupe (0 / 1 / 2)
    axes: Optional[Dict[str, object]] = None     # factored candidate set (candidate_axes): no per-candidate arrays
    cand_first: int = 0                          # product index of the batch's first candidate

    def h2d_bytes(self) -> int:
        return int(sum(a.nbytes for a in self.arrays.values()))

    def max_radius(self) -> float:
        if "cand_R" in self.arrays:
            return float(self.arrays["cand_R"].max())
        if self.axes is not None and "R" in self.axes:
            return float(self.axes["R"].max())
        return float(self.vehicle.min_turn_radius)


def _obstacle_tables(obstacles, F: int, W: float, arrays: Dict[str, np.ndarray]):
    """Obstacles (mlp3:600-609), one polygon list per field, as the flattened fcpp_batch tables + D2 round-buffer
    moments, added to ``arrays`` (nothing when there is no obstacle).  -> (max vertices, max polygons) of a field."""
    max_v = max_p = 0
    if obstacles is not None and any(len(o) for o in obstacles):
        if len(obstacles) != F:
            raise ValueError("obstacles must have one (possibly empty) polygon list per field")
        poly_start = [0]
        vert_start = [0]
        verts: List[Sequence[float]] = []
        moms = []
        for polys in obstacles:
            nv_field = 0
            for poly in polys:
                pts = [tuple(map(float, p)) for p in poly]
                verts.extend(pts)
                nv_field += len(pts)
                vert_start.append(len(verts))
                moms.append(G.round_buffer_moments(pts, W / 2))
            poly_start.append(len(vert_start) - 1)
            max_v = max(max_v, nv_field)
            max_p = max(max_p, len(polys))
        arrays["obs_poly_start"] = np.asarray(poly_start, dtype=np.int32)
        arrays["obs_vert_start"] = np.asarray(vert_start, dtype=np.int32)
        arrays["obs_verts"] = np.asarray(verts, dtype=np.float64).reshape(-1, 2)
        arrays["obs_moments"] = np.asarray(moms, dtype=np.float64).reshape(-1, 3)
    return max_v, max_p


def prepare_batch(fields, vehicle: VehicleParams, candidates: Optional[Dict[str, np.ndarray]] = None,
                  obstacles: Optional[Sequence[Sequence[Sequence[Sequence[float]]]]] = None,
                  start_points: Optional[np.ndarray] = None, grid_h: float = 0.1,
                  coverage: bool = True, turn_model: str = "arc", clothoid_share: float = 0.5) -> PreparedBatch:
    """FP64 host set-up (A2).  ``fields`` [F,4,2] convex CCW quads; ``obstacles`` = per field a
    list of polygons; ``candidates`` = dict with ``field_id`` and optional ``heading`` (rad),
    ``R``, ``start_corner`` arrays of length B (default: one candidate per field with the
    reference's defaults); ``start_points`` [B,2] makes the pass order follow mlp3:631-668."""
    fv = np.ascontiguousarray(np.asarray(fields, dtype=np.float64).reshape(-1, 4, 2))
    F = len(fv)
    W = float(vehicle.working_width)
    # ---- per field: bbox extents (mlp3:120-122), reverse-fill permission bits (mlp3:224-242) ----
    ext = np.stack([fv[:, :, 0].max(1) - fv[:, :, 0].min(1), fv[:, :, 1].max(1) - fv[:, :, 1].min(1)], axis=1)
    ang = G.corner_angles_deg(fv)
    fflags = ((ang >= 60).astype(np.int32) << np.arange(4, dtype=np.int32)).sum(axis=1).astype(np.int32)
    arrays = {"field_verts": fv, "field_extent": np.ascontiguousarray(ext), "field_flags": fflags}
    axes = None
    cand_first = 0

    def rot_of(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        return (np.ascontiguousarray(np.stack([np.cos(-a), np.sin(-a), np.cos(a), np.sin(a)], axis=1)),
                np.abs(a) > ROT_THRESHOLD)

    def field_rot():
        # the reference's heading is a property of the field (direction of edge 0, mlp3:244-263)
        e0 = fv[:, 1, :] - fv[:, 0, :]
        return rot_of(np.arctan2(e0[:, 1], e0[:, 0]))

    if is_axes(candidates):
        # ---- factored candidate set: per AXIS value what the explicit form computes per candidate ----
        axes = candidates
        if int(axes["n_fields"]) != F:
            raise ValueError("candidate axes were made for another number of fields")
        if start_points is not None:
            raise ValueError("start_points need explicit candidate arrays (make_candidates)")
        per = axes_per_field(axes)
        cand_first, hi = axes.get("range", (0, F * per))
        if not (0 <= cand_first <= hi <= F * per):
            raise ValueError("candidate range beyond the product of the axes")
        B = int(hi - cand_first)
        if "heading" in axes:
            rot, rotated = rot_of(axes["heading"])
            arrays["ax_heading_rot"] = rot
            arrays["ax_heading_flags"] = (rotated.astype(np.int32) * _lib.FLAG_ROTATED).astype(np.int32)
        else:
            rot, rotated = field_rot()
            arrays["field_rot"] = rot
            arrays["field_rot_flags"] = (rotated.astype(np.int32) * _lib.FLAG_ROTATED).astype(np.int32)
        if "R" in axes:
            arrays["ax_radii"] = axes["R"]
            arrays["ax_radius_flags"] = (G.gap_gate(axes["R"], W).astype(np.int32) * _lib.FLAG_GAP_GATE).astype(np.int32)
        if "start_corner" in axes:
            c = axes["start_corner"]
            if c.min() < 0 or c.max() > 3:
                raise ValueError("start_corner must be 0..3")
            arrays["ax_corners"] = c
        dedupe = B > F and ("heading" in axes or "start_corner" in axes)
        if dedupe and "heading" in axes and B >= 4 * F:
            dedupe = 2          # a heading search: few coverage representatives (fcpp_batch.cover_dedupe = 2)
    else:
        if candidates is None:
            candidates = {"field_id": np.arange(F, dtype=np.int32)}
        fid = np.ascontiguousarray(candidates["field_id"], dtype=np.int32)
        B = len(fid)
        if B and (fid.min() < 0 or fid.max() >= F):
            raise ValueError("candidate field_id out of range")
        R = np.ascontiguousarray(candidates.get("R", np.full(B, vehicle.min_turn_radius)), dtype=np.float64)
        if "heading" in candidates:
            rot, rotated = rot_of(candidates["heading"])
        else:
            rot_f, rotated_f = field_rot()            # trig per field, gathered
            rot = np.take(rot_f, fid, axis=0)
            rotated = np.take(rotated_f, fid)
        if "start_corner" in candidates:
            c = np.asarray(candidates["start_corner"], dtype=np.int32)
            if B and (c.min() < 0 or c.max() > 3):
                raise ValueError("start_corner must be 0..3")
            # corner c in {0: LB, 1: RB, 2: RT, 3: LT}: reverse order iff c in {2, 3}, start from the right
            # iff c in {1, 2} (mlp3:650-658)
            hi_ = c >> 1
            flags = c | (hi_ * _lib.FLAG_REVERSE_ORDER) | (((c ^ hi_) & 1) * _lib.FLAG_START_FROM_RIGHT)
            flags = flags.astype(np.int32, copy=False)
        else:
            flags = np.zeros(B, dtype=np.int32)
        flags |= rotated.astype(np.int32) * _lib.FLAG_ROTATED
        flags |= G.gap_gate(R, W).astype(np.int32) * _lib.FLAG_GAP_GATE
        arrays.update({"cand_field": fid, "cand_R": R, "cand_rot": np.ascontiguousarray(rot), "cand_flags": flags})
        if start_points is not None:
            sp = np.ascontiguousarray(start_points, dtype=np.float64).reshape(B, 2)
            use = ~np.isnan(sp[:, 0])
            flags |= np.where(use, _lib.FLAG_START_POINT, 0).astype(np.int32)
            arrays["cand_start"] = np.where(use[:, None], sp, 0.0)
        dedupe = B > F and ("heading" in candidates or "start_corner" in candidates)
        if dedupe and "heading" in candidates and B >= 4 * F:
            dedupe = 2          # a heading search: few coverage representatives (fcpp_batch.cover_dedupe = 2)
    max_v, max_p = _obstacle_tables(obstacles, F, W, arrays)
    if turn_model not in ("arc", "clothoid", "omega"):
        raise ValueError("turn_model must be 'arc' (the reference's sampled arcs), 'clothoid' or 'omega'")
    return PreparedBatch(vehicle, F, B, arrays, max_v, max_p, float(grid_h), bool(coverage), turn_model,
                         float(clothoid_share), dedupe=dedupe, axes=axes, cand_first=int(cand_first))


class DeviceBatch:
    """A PreparedBatch resident in HBM + its ctypes descriptor."""

    def __init__(self, pb: PreparedBatch, dev: torch.device, pin: bool = True, slot: int = 0):
        self.pb = pb
        self.dev = dev
        self.slot = slot   # which handle / staging buffers / (by convention) stream this batch uses
        self.t = (_pack_to_dev(pb.arrays, dev, slot) if pin
                  else {k: _to_dev(v, dev, False) for k, v in pb.arrays.items()})
        v = pb.vehicle
        b = _lib.Batch()
        b.vehicle = _lib.Vehicle(v.working_width, v.max_work_speed_kmh, v.max_headland_speed_kmh,
                                 v.headland_turn_speed_kmh, v.max_lateral_accel, v.max_longitudinal_accel,
                                 v.safety_factor, 2.5)
        b.n_fields = pb.n_fields
        b.n_cand = pb.n_cand
        for name in ("field_verts", "field_extent", "field_flags", "obs_poly_start", "obs_vert_start",
                     "obs_verts", "obs_moments", "cand_field", "cand_R", "cand_rot", "cand_flags", "cand_start"):
            t = self.t.get(name)
            setattr(b, name, t.data_ptr() if t is not None else None)
        b.max_obs_verts = pb.max_obs_verts
        b.max_obs_polys = pb.max_obs_polys
        b.grid_h = pb.grid_h
        b.do_coverage = 1 if pb.coverage else 0
        b.turn_model = {"arc": 0, "clothoid": 1, "omega": 2}[pb.turn_model]
        # the headings of a field repeat its headland (hence its coverage), its start corners repeat the
        # corner-window verification: identical coverage work is done once per group on the device
        b.cover_dedupe = int(pb.dedupe)
        b.clothoid_share = pb.clothoid_share
        if pb.axes is not None:
            ax = pb.axes
            b.n_ax_headings = len(ax["heading"]) if "heading" in ax else 0
            b.n_ax_radii = len(ax["R"]) if "R" in ax else 0
            b.n_ax_corners = len(ax["start_corner"]) if "start_corner" in ax else 0
            b.ax_default_radius = float(v.min_turn_radius)
            b.ax_default_radius_flags = _lib.FLAG_GAP_GATE if bool(G.gap_gate(np.array([v.min_turn_radius]),
                                                                              float(v.working_width))[0]) else 0
            b.cand_first = pb.cand_first
            for name in ("ax_heading_rot", "ax_heading_flags", "ax_radii", "ax_radius_flags", "ax_corners",
                         "field_rot", "field_rot_flags"):
                t = self.t.get(name)
                setattr(b, name, t.data_ptr() if t is not None else None)
        self.c = b


@dataclass
class BatchResult:
    """Per-candidate summaries (host numpy structured array, dtype _lib.SUMMARY_DTYPE), the
    per-field argmin, and — in ``outputs='paths'`` mode — device-resident paths."""
    summary: np.ndarray
    best_cand: np.ndarray          # [F] int64 global candidate index (-1: no valid candidate)
    best_cost: np.ndarray          # [F] float64
    n_fields: int
    offsets: Optional[np.ndarray] = None        # [B+1] int64 (paths mode)
    d_path: Optional[torch.Tensor] = None       # [total, 2] float64 on device
    d_speeds: Optional[torch.Tensor] = None     # [total] float64 km/h on device
    d_curvature: Optional[torch.Tensor] = None
    d_summary: Optional[torch.Tensor] = None
    cand_base: int = 0
    extras: Dict = dc_field(default_factory=dict)
    # plan_batch(..., winners=True): field -> (path [n,2], speeds [n] km/h, n_main) of the field's best candidate, on
    # the host (in a distributed run: the fields whose winner this rank owns)
    winner_paths: Optional[Dict[int, tuple]] = None
    # plan_batch(..., select=Selection(top_k=k)): per field the k best eligible candidates (global indices, -1 = none),
    # their costs (+inf = none) and summary records (zeros = none); best_cand / best_cost are column 0
    topk_cand: Optional[np.ndarray] = None      # [F, k] int64
    topk_cost: Optional[np.ndarray] = None      # [F, k] float64
    topk_summary: Optional[np.ndarray] = None   # [F, k] SUMMARY_DTYPE
    # plan_batch(..., obstacle_sweep=True): per candidate the segments that drive through the obstacle region and the
    # metres inside, per layer (include/fcpp.h fcpp_sweep)
    sweep: Optional[np.ndarray] = None          # [B] SWEEP_DTYPE
    # plan_batch(..., field_coverage=True): per candidate the D3 counts and the cells of the headland band and of the
    # whole field with those the plan covers (include/fcpp.h fcpp_path_cover)
    field_cover: Optional[np.ndarray] = None    # [B] PATH_COVER_DTYPE

    def path(self, b: int):
        """(path [n,2], speeds [n], n_main) of local candidate ``b`` copied to the host."""
        if self.d_path is None:
            raise ValueError("plan_batch was run with outputs='summary'")
        o0, o1 = int(self.offsets[b]), int(self.offsets[b + 1])
        return (self.d_path[o0:o1].cpu().numpy(), self.d_speeds[o0:o1].cpu().numpy(),
                int(self.summary["n_main"][b]))


class BatchBuffers:
    """Device output buffers of one batch shape, reusable across calls (steady-state serving:
    no allocation, no readback, no synchronisation inside the step)."""

    def __init__(self, dev: torch.device, n_cand: int, n_fields: int, total_points: int = 0,
                 want_curvature: bool = False, path_storage=None):
        """``path_storage`` = (d_path [total, 2], d_spd [total], d_kap [total] | None): views of a larger
        allocation to use instead of new tensors."""
        self.dev = dev
        self.n_cand, self.n_fields, self.total_points = n_cand, n_fields, total_points
        self.d_sum = torch.empty(max(n_cand, 1) * _lib.SUMMARY_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        self.d_cost = self.d_best = None
        self.rank_k(1)
        self.d_off = self.d_path = self.d_spd = self.d_kap = None
        self.d_sweep = None          # [B] fcpp_sweep records of the last batch run with obstacle_sweep=True
        self.d_fcov = None           # [B] fcpp_path_cover records of the last batch run with field_coverage=True
        self.speculative = False     # sized from remembered maxima (_Hints), not from this batch's layout pass
        if total_points > 0:
            self.d_off = torch.empty(n_cand + 1, dtype=torch.int64, device=dev)
            if path_storage is not None:
                self.d_path, self.d_spd, self.d_kap = path_storage
            else:
                self.d_path = torch.empty((total_points, 2), dtype=torch.float64, device=dev)
                self.d_spd = torch.empty(total_points, dtype=torch.float64, device=dev)
                if want_curvature:
                    self.d_kap = torch.empty(total_points, dtype=torch.float64, device=dev)

    def rank_k(self, k: int):
        """Size the per-field ranking for k entries per field: ``d_cost`` [F, k] (flat) then ``d_best`` [F, k] (global
        candidate indices), back to back in ONE allocation (the multi-GPU merge all-gathers both at once); at k = 1
        they are the per-field best.  Reallocated only when k changes."""
        nfk = max(self.n_fields, 1) * int(k)
        if self.d_cost is None or self.d_cost.numel() != nfk:
            ranking = torch.empty(2 * nfk, dtype=torch.int64, device=self.dev)
            self.d_cost, self.d_best = ranking[:nfk].view(torch.float64), ranking[nfk:]


def corner_grids(words: np.ndarray, g: int) -> np.ndarray:
    """[4, g, g] bool occupancy grids (grid[c][j, i] = lattice point (i, j) of corner c, mlp3:1477) from one
    candidate's ``corner_bits`` words (fcpp_outputs.corner_bits layout)."""
    rw = (g + 31) // 32
    w = np.ascontiguousarray(words[:4 * g * rw], dtype=np.uint32).reshape(4, g, rw)
    bits = np.unpackbits(w.view(np.uint8).reshape(4, g, rw * 4), axis=2, bitorder="little")
    return bits[:, :, :g].astype(bool)


class _Hints:
    """Sizes of earlier batches of the same shape (same fields, vehicle width, grid, candidate count): the longest
    plan, the longest headland, the total number of points.  A batch that finds its shape here is launched WITHOUT
    the layout pass's synchronous read-back — staging sized by the remembered maxima, path buffers by the remembered
    total (fcpp_outputs.path_capacity guards them).  A candidate that needs more is flagged FCPP_CAND_TOO_LARGE /
    FCPP_CAND_GRID_TOO_LARGE by the kernels; the caller (PendingBatch.result) then runs the batch once more with
    sizes from its own layout pass, so results never depend on the cache."""
    _c: Dict[tuple, list] = {}

    @staticmethod
    def key(db: "DeviceBatch", outputs: str, want_curvature: bool) -> tuple:
        pb = db.pb
        fv = pb.arrays["field_verts"]
        return (db.dev.index, outputs, bool(want_curvature), pb.n_fields, pb.n_cand, float(fv.sum()) if fv.size else 0.0,
                float(pb.vehicle.working_width), pb.grid_h, pb.turn_model, pb.coverage, pb.max_obs_verts)

    @classmethod
    def get(cls, key):
        return cls._c.get(key)

    @classmethod
    def update(cls, key, max_points: int, max_head: int, total: int):
        e = cls._c.get(key)
        if e is None:
            if len(cls._c) > 64:
                cls._c.clear()
            cls._c[key] = [int(max_points), int(max_head), int(total)]
        else:
            e[0], e[1], e[2] = max(e[0], int(max_points)), max(e[1], int(max_head)), max(e[2], int(total))

    @classmethod
    def drop(cls, key):
        cls._c.pop(key, None)


def _launch_device_batch(db: DeviceBatch, outputs: str, want_curvature: bool, selection: Selection, cand_base: int,
                         buffers: Optional["BatchBuffers"], path_alloc=None, corner_bits: bool = False,
                         speculate: bool = False, sweep: bool = False, field_cover: bool = False):
    """Enqueue layout, prefix sum, plan, coverage and ranking kernels of one batch on torch's current
    stream.  Returns (buffers, offsets or None).  Without ``buffers`` the path storage is sized from
    the layout pass (one small synchronous read-back) — or, with ``speculate`` and a batch of this shape seen
    before, from the remembered sizes with no synchronisation at all (``buffers.speculative`` is then True and the
    caller must check the status flags, see ``_Hints``); ``path_alloc(total) -> BatchBuffers | None`` lets the
    caller provide the storage.  ``selection``: how fcpp_field_select ranks each field's candidates into
    buffers.d_cost / d_best.  ``sweep``: also the segment-level obstacle sweep of every candidate
    (fcpp_obstacle_sweep) into buffers.d_sweep.  ``field_cover`` (paths mode): also the whole-field and headland-band
    coverage of the materialised paths (fcpp_plan_coverage) into buffers.d_fcov."""
    if outputs not in ("summary", "paths"):
        raise ValueError("outputs must be 'summary' or 'paths'")
    dev = db.dev
    h = _lib.handle(dev.index, db.slot)
    L = h.lib
    B, F = db.pb.n_cand, db.pb.n_fields
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    hint_key = _Hints.key(db, outputs, want_curvature) if buffers is None and B > 0 else None
    hint = _Hints.get(hint_key) if (speculate and hint_key is not None and path_alloc is None) else None
    with torch.cuda.device(dev):
        out = _lib.Outputs()
        offsets = None
        if hint is not None and hint[0] > 0 and hint[1] > 0:
            db.c.max_points_hint, db.c.max_head_points_hint = hint[0], hint[1]
            total = max(hint[2], 1) if outputs == "paths" else 0
            buffers = BatchBuffers(dev, B, F, total, want_curvature)
            buffers.speculative = True
            if outputs == "paths":
                h.check(L.fcpp_layout(h.h, C.byref(db.c), None, buffers.d_off.data_ptr(), stream))
                out.path_capacity = total
        elif buffers is None:
            db.c.max_points_hint = 0
            db.c.max_head_points_hint = 0
            total = 0
            if outputs == "paths":
                d_off = torch.empty(B + 1, dtype=torch.int64, device=dev)
                h.check(L.fcpp_layout(h.h, C.byref(db.c), None, d_off.data_ptr(), stream))
                # the layout pass's own read-back carries the total; the offsets come back with the summaries
                total = int(L.fcpp_last_total_points(h.h))
                if total < 0:
                    offsets = d_off.cpu().numpy()
                    total = int(offsets[-1])
                total = max(total, 1)
            buffers = path_alloc(total) if path_alloc is not None else None
            if buffers is None:
                buffers = BatchBuffers(dev, B, F, total, want_curvature)
            if outputs == "paths":
                buffers.d_off = d_off
        else:
            db.c.max_points_hint = int(getattr(db, "max_points", 0))
            db.c.max_head_points_hint = int(getattr(db, "max_head_points", 0))
            if outputs == "paths":
                if buffers.d_off is None:
                    raise ValueError("buffers were allocated without path storage")
                h.check(L.fcpp_layout(h.h, C.byref(db.c), None, buffers.d_off.data_ptr(), stream))
        out.summary = buffers.d_sum.data_ptr()
        if corner_bits:
            # occupancy bits of the four verification corner windows (mlp3:1503-1510 'grid'), sized by the largest R
            g = int(2 * db.pb.max_radius() / 0.1) if B else 1
            stride = 4 * g * ((g + 31) // 32)
            if getattr(buffers, "d_cbits", None) is None or buffers.d_cbits.numel() < B * stride:
                buffers.d_cbits = torch.zeros(max(B * stride, 1), dtype=torch.int32, device=dev)
            buffers.cbits_stride = stride
            out.corner_bits = buffers.d_cbits.data_ptr()
            out.corner_bits_stride = stride
        if outputs == "paths":
            out.offsets = buffers.d_off.data_ptr()
            out.path_xy = buffers.d_path.data_ptr()
            out.speeds_kmh = buffers.d_spd.data_ptr()
            if buffers.d_kap is not None:
                out.curvature = buffers.d_kap.data_ptr()
        h.check(L.fcpp_plan_batch(h.h, C.byref(db.c), C.byref(out), stream))
        if sweep:
            nb = max(B, 1) * _lib.SWEEP_DTYPE.itemsize
            if buffers.d_sweep is None or buffers.d_sweep.numel() < nb:
                buffers.d_sweep = torch.empty(nb, dtype=torch.uint8, device=dev)
            h.check(L.fcpp_obstacle_sweep(h.h, C.byref(db.c), buffers.d_sweep.data_ptr(), stream))
        if field_cover:
            nb = max(B, 1) * _lib.PATH_COVER_DTYPE.itemsize
            if buffers.d_fcov is None or buffers.d_fcov.numel() < nb:
                buffers.d_fcov = torch.empty(nb, dtype=torch.uint8, device=dev)
            h.check(L.fcpp_plan_coverage(h.h, C.byref(db.c), C.byref(out), buffers.d_fcov.data_ptr(), stream))
        if db.c.max_points_hint == 0:
            db.max_points = int(L.fcpp_last_max_points(h.h))
            db.max_head_points = int(L.fcpp_last_max_head_points(h.h))
            if hint_key is not None:
                _Hints.update(hint_key, db.max_points, db.max_head_points, buffers.total_points)
        cf = db.t.get("cand_field")     # factored sets: the library's candidate records carry the field
        buffers.rank_k(selection.top_k)
        sc = selection.c_struct(db.pb.grid_h)
        h.check(L.fcpp_field_select(h.h, buffers.d_sum.data_ptr(), cf.data_ptr() if cf is not None else None, B, F,
                                    C.byref(sc), cand_base, buffers.d_cost.data_ptr(), buffers.d_best.data_ptr(),
                                    stream))
    return buffers, offsets


class _PendingFetch:
    """The read-back of a launched batch, enqueued but not waited for."""
    __slots__ = ("db", "buffers", "outputs", "offsets", "cand_base", "hv", "lay", "win", "hwin", "event", "o_sweep",
                 "o_fcov")


def _enqueue_fetch(db: DeviceBatch, buffers: "BatchBuffers", outputs: str, offsets, copy_summary: bool,
                   cand_base: int, win: Optional[torch.Tensor] = None, sweep: bool = False,
                   field_cover: bool = False) -> _PendingFetch:
    """Enqueue the copies of summaries + the per-field ranking (+ offsets) (+ ``win``: the winners' records and
    flag-count word of a sharded batch, see dist.gather_winner_records) (+ ``sweep``: the obstacle sweep records)
    (+ ``field_cover``: the field coverage records)
    into ONE pooled pinned buffer on torch's current stream and record an event behind them; nothing is waited for."""
    dev = db.dev
    B, F = db.pb.n_cand, db.pb.n_fields
    k = buffers.d_cost.numel() // max(F, 1)     # entries per field of the ranking
    pf = _PendingFetch()
    with torch.cuda.device(dev):
        nb_sum = B * _lib.SUMMARY_DTYPE.itemsize if copy_summary else 0
        need_off = outputs == "paths" and offsets is None
        o_cost = (nb_sum + 255) & ~255
        o_best = o_cost + ((F * k * 8 + 255) & ~255)
        o_off = o_best + ((F * k * 8 + 255) & ~255)
        total_out = o_off + ((B + 1) * 8 if need_off else 0)
        o_win = (total_out + 255) & ~255
        if win is not None:
            total_out = o_win + win.numel()
        o_sweep = (total_out + 255) & ~255
        nb_sweep = B * _lib.SWEEP_DTYPE.itemsize if sweep else 0
        if sweep:
            total_out = o_sweep + nb_sweep
        o_fcov = (total_out + 255) & ~255
        nb_fcov = B * _lib.PATH_COVER_DTYPE.itemsize if field_cover else 0
        if field_cover:
            total_out = o_fcov + nb_fcov
        ho, hv = _ResultPool.get(total_out)
        # the copies run on a COPY stream behind an event of the launching stream: the next batch's kernels (already
        # enqueued by a pipelining caller) must not wait for PCIe — at 737 280 candidates the 130 MB of summaries
        # share the link with the 360 MB of the previous batch's winners' paths
        # (small read-backs stay on the launching stream: the extra stream costs more than it hides.)  The device
        # buffers stay referenced by the pending fetch / the result until the event has been waited for, so the
        # allocator cannot hand them out while the copy runs.
        main = torch.cuda.current_stream(dev)
        cs = _copy_stream(dev) if total_out >= (8 << 20) else main
        if cs is not main:
            done = torch.cuda.Event()
            done.record(main)
            cs.wait_event(done)
        with torch.cuda.stream(cs):
            if nb_sum:
                ho[:nb_sum].copy_(buffers.d_sum[:nb_sum], non_blocking=True)
            if F:
                ho[o_cost:o_cost + F * k * 8].view(torch.float64).copy_(buffers.d_cost[:F * k], non_blocking=True)
                ho[o_best:o_best + F * k * 8].view(torch.int64).copy_(buffers.d_best[:F * k], non_blocking=True)
            if need_off:
                ho[o_off:o_off + (B + 1) * 8].view(torch.int64).copy_(buffers.d_off[:B + 1], non_blocking=True)
            if win is not None:
                ho[o_win:o_win + win.numel()].copy_(win, non_blocking=True)
            if nb_sweep:
                ho[o_sweep:o_sweep + nb_sweep].copy_(buffers.d_sweep[:nb_sweep], non_blocking=True)
            if nb_fcov:
                ho[o_fcov:o_fcov + nb_fcov].copy_(buffers.d_fcov[:nb_fcov], non_blocking=True)
            pf.event = torch.cuda.Event()
            pf.event.record(cs)
    pf.db, pf.buffers, pf.outputs, pf.offsets, pf.cand_base = db, buffers, outputs, offsets, cand_base
    pf.hv, pf.lay = hv, (nb_sum, need_off, o_cost, o_best, o_off, k)
    pf.win, pf.hwin = win, (hv[o_win:o_win + win.numel()] if win is not None else None)
    pf.o_sweep = (o_sweep, B) if sweep else None
    pf.o_fcov = (o_fcov, B) if field_cover else None
    return pf


def _finish_fetch(pf: _PendingFetch, ranked: bool) -> "BatchResult":
    """Wait for the read-back of ``_enqueue_fetch`` (ONE synchronisation, on its event) and assemble the result:
    its arrays are views of the read-back's own pooled buffer.  ``ranked``: the caller asked for the ranking
    (``topk_cand`` / ``topk_cost``); ``best_cand`` / ``best_cost`` are its first column either way."""
    db, buffers, offsets, hv = pf.db, pf.buffers, pf.offsets, pf.hv
    B, F = db.pb.n_cand, db.pb.n_fields
    nb_sum, need_off, o_cost, o_best, o_off, k = pf.lay
    pf.event.synchronize()
    summary = hv[:nb_sum].view(_lib.SUMMARY_DTYPE)[:B] if nb_sum else np.zeros(0, dtype=_lib.SUMMARY_DTYPE)
    topk_cost = hv[o_cost:o_cost + F * k * 8].view(np.float64).reshape(F, k)
    topk_cand = hv[o_best:o_best + F * k * 8].view(np.int64).reshape(F, k)
    if need_off:
        offsets = hv[o_off:o_off + (B + 1) * 8].view(np.int64)
    res = BatchResult(summary=summary, best_cand=np.ascontiguousarray(topk_cand[:, 0]),
                      best_cost=np.ascontiguousarray(topk_cost[:, 0]), n_fields=F, offsets=offsets,
                      d_path=buffers.d_path, d_speeds=buffers.d_spd, d_curvature=buffers.d_kap,
                      d_summary=buffers.d_sum, cand_base=pf.cand_base)
    if ranked:
        res.topk_cand, res.topk_cost = topk_cand, topk_cost
    if pf.o_sweep is not None:
        o, n = pf.o_sweep
        res.sweep = hv[o:o + n * _lib.SWEEP_DTYPE.itemsize].view(_lib.SWEEP_DTYPE)
    if pf.o_fcov is not None:
        o, n = pf.o_fcov
        res.field_cover = hv[o:o + n * _lib.PATH_COVER_DTYPE.itemsize].view(_lib.PATH_COVER_DTYPE)
    res.extras["buffers"] = buffers
    return res


_side_streams: Dict[int, "torch.cuda.Stream"] = {}
_copy_streams: Dict[int, "torch.cuda.Stream"] = {}


def _copy_stream(dev: torch.device) -> "torch.cuda.Stream":
    """The stream the result read-back of a batch runs on (see _enqueue_fetch)."""
    st = _copy_streams.get(dev.index)
    if st is None:
        st = _copy_streams[dev.index] = torch.cuda.Stream(device=dev, priority=-1)
    return st


def _side_stream(dev: torch.device) -> "torch.cuda.Stream":
    """A second stream per device for the winners' read-back of a finished batch: it must not queue behind the
    kernels of the NEXT batch, which a pipelining caller has already launched on the main stream.  HIGH priority:
    the small kernels of the winners' batch are dispatched ahead of the remaining CTAs of a 737 280-CTA grid of the
    main stream — at default priority they waited until that grid had been dispatched completely (33 ms), the host
    sat in result() meanwhile and the GPU idled 8 ms per step before the next submit (tools/pipeline_trace.py)."""
    st = _side_streams.get(dev.index)
    if st is None:
        st = _side_streams[dev.index] = torch.cuda.Stream(device=dev, priority=-1)
    return st


def _read_back_paths(d_path: torch.Tensor, d_speeds: torch.Tensor, spans):
    """The point ranges ``spans`` [(a, b), ...] of a device path and its speeds, back to back in one pooled pinned
    buffer: async copies on torch's current stream, ONE synchronisation.  -> (path [n, 2], speeds [n]) numpy views."""
    tot = sum(b - a for a, b in spans)
    ho, hv = _ResultPool.get(tot * 24 + 256)
    hp = ho[:tot * 16].view(torch.float64).view(tot, 2)
    hs = ho[tot * 16:tot * 24].view(torch.float64)
    at = 0
    for a, b in spans:
        hp[at:at + b - a].copy_(d_path[a:b], non_blocking=True)
        hs[at:at + b - a].copy_(d_speeds[a:b], non_blocking=True)
        at += b - a
    torch.cuda.current_stream(d_path.device).synchronize()
    return hv[:tot * 16].view(np.float64).reshape(tot, 2), hv[tot * 16:tot * 24].view(np.float64)


def fetch_winner_paths(db: DeviceBatch, res: BatchResult, outputs: str, best_cand: Optional[np.ndarray] = None,
                       slot: Optional[int] = None) -> int:
    """Bring the path and the speed profile of every field's best candidate to the host
    (``res.winner_paths``); returns the bytes copied device -> host.  ``best_cand`` (default: the batch's own
    argmin) holds GLOBAL candidate indices; winners outside this batch's range (other ranks' candidates in a
    distributed run) are skipped.

    outputs='paths' and a few winners: slices of the materialised paths, one synchronisation.  Otherwise (the
    search configurations, which run summary-only) the winners are planned again as their own small batch
    with materialised paths — the candidate arrays are slices of the prepared batch, coverage off.  ``slot``: the
    handle / staging slot of that second batch (a caller that runs this on a side stream next to batches in flight
    on the main stream must not share their handle's workspace)."""
    dev = db.dev
    B = db.pb.n_cand
    slot = db.slot if slot is None else slot
    best = res.best_cand if best_cand is None else best_cand
    own = np.nonzero((best >= res.cand_base) & (best < res.cand_base + B))[0]
    res.winner_paths = {}
    if len(own) == 0:
        return 0
    local = (best[own] - res.cand_base).astype(np.int64)
    with torch.cuda.device(dev):
        if outputs == "paths" and len(own) <= 16 and res.offsets is not None:
            o0, o1 = res.offsets[local], res.offsets[local + 1]
            P, S = _read_back_paths(res.d_path, res.d_speeds, [(int(a), int(b)) for a, b in zip(o0, o1)])
            offs = np.concatenate([[0], np.cumsum(o1 - o0)])
            nbytes = len(S) * 24
        else:
            if db.pb.axes is not None:
                # the winners of a factored set as explicit candidates (a few values per field from the axes)
                keep = {k: v for k, v in db.pb.arrays.items() if k.startswith(("field_", "obs_")) and
                        k not in ("field_rot", "field_rot_flags")}
                pbx = prepare_batch(db.pb.arrays["field_verts"], db.pb.vehicle,
                                    expand_axes(db.pb.axes, db.pb.cand_first + local), None, None, db.pb.grid_h, False,
                                    db.pb.turn_model, db.pb.clothoid_share)
                arrays = dict(pbx.arrays)
                arrays.update(keep)
            else:
                arrays = dict(db.pb.arrays)
                for k in ("cand_field", "cand_R", "cand_rot", "cand_flags", "cand_start"):
                    if k in arrays:
                        arrays[k] = np.ascontiguousarray(arrays[k][local])
            pbw = PreparedBatch(db.pb.vehicle, db.pb.n_fields, len(local), arrays, db.pb.max_obs_verts,
                                db.pb.max_obs_polys, db.pb.grid_h, False, db.pb.turn_model, db.pb.clothoid_share, False)
            dbw = DeviceBatch(pbw, dev, slot=slot)
            rw = run_device_batch(dbw, "paths", copy_summary=False)
            tot = int(rw.offsets[-1])
            P, S = _read_back_paths(rw.d_path, rw.d_speeds, [(0, tot)])
            offs = rw.offsets
            nbytes = tot * 24 + (len(local) + 1) * 8 + 16 * db.pb.n_fields
            res.extras["h2d_bytes"] = res.extras.get("h2d_bytes", 0) + pbw.h2d_bytes()
    nm = res.summary["n_main"] if len(res.summary) == B else None
    for k, f in enumerate(own):
        a, b = int(offs[k]), int(offs[k + 1])
        n_main = int(nm[local[k]]) if nm is not None else -1
        res.winner_paths[int(f)] = (P[a:b], S[a:b], n_main)
    return nbytes


_SIZE_FLAGS = 8 | 16      # FCPP_CAND_TOO_LARGE | FCPP_CAND_GRID_TOO_LARGE (include/fcpp.h)


class PendingBatch:
    """A batch whose kernels and read-back are enqueued (``plan_batch(..., wait=False)``); ``result()`` waits for
    them and returns the BatchResult.  A caller that submits batch k+1 before asking for the result of batch k
    overlaps its host work (set-up, packed copy, launches) with the kernels of batch k:

        pend = plan_batch(..., wait=False)
        for next_candidates in search:
            nxt = plan_batch(..., candidates=next_candidates, wait=False)
            res = pend.result()
            pend = nxt

    A sharded batch (``plan_batch(..., distributed=True)``) is collected the same way on every rank; its
    ``result()`` is COLLECTIVE in one case only: when some rank's remembered launch sizes did not fit its shard,
    all ranks repeat the batch together."""

    def __init__(self, db, pf, outputs, want_curvature, selection, ranked, cand_base, copy_summary, winners,
                 corner_bits, speculate, shard, sweep=False, field_cover=False):
        self.db, self.pf, self.outputs = db, pf, outputs
        self.args = (want_curvature, selection, ranked, cand_base, copy_summary, winners, corner_bits, sweep,
                     field_cover)
        self.speculate, self.shard = speculate, shard
        self._res = None

    def __del__(self):
        # an abandoned batch: its read-back may still be in flight into pooled pinned memory / out of buffers that
        # the allocator is about to hand out again — wait for it before letting go
        try:
            if self._res is None and self.pf is not None:
                self.pf.event.synchronize()
        except Exception:
            pass

    def result(self) -> "BatchResult":
        if self._res is not None:
            return self._res
        db, pf, outputs = self.db, self.pf, self.outputs
        want_curvature, selection, ranked, cand_base, copy_summary, winners, corner_bits, sweep, field_cover = self.args
        buffers = pf.buffers
        B, F = db.pb.n_cand, db.pb.n_fields
        k = selection.top_k
        rec = _lib.SUMMARY_DTYPE.itemsize
        res = _finish_fetch(pf, ranked)
        if self.shard is None:
            redo = buffers.speculative and (not copy_summary or (res.summary["status"] & _SIZE_FLAGS).any())
        else:
            # the number of flagged candidates OF ALL RANKS: every rank reads the same word and decides alike, also
            # a rank that had no remembered sizes itself
            redo = self.speculate and int(pf.hwin[F * k * rec:F * k * rec + 4].view(np.int32)[0]) != 0
        if redo:
            # remembered sizes (see _Hints) did not fit this batch, or cannot be checked: once more, sized from its
            # own layout pass.  (A batch with candidates that are genuinely too large takes this path too and comes
            # back with the same flags.)
            _Hints.drop(_Hints.key(db, outputs, want_curvature))
            self._res = _run_device_batch(db, outputs, want_curvature, selection, ranked, cand_base, copy_summary,
                                          buffers=None, fetch=True, winners=winners, corner_bits=corner_bits,
                                          speculate=False, wait=True, shard=self.shard, obstacle_sweep=sweep,
                                          field_coverage=field_cover)
            return self._res
        if corner_bits:   # [B, stride] words on the device; batch.corner_grids() unpacks one candidate's
            res.extras["corner_bits"] = buffers.d_cbits[:B * buffers.cbits_stride].view(B, -1)
        res.extras["h2d_bytes"] = db.pb.h2d_bytes()
        res.extras["d2h_bytes"] = len(res.summary) * rec + 16 * F * k + ((B + 1) * 8 if outputs == "paths" else 0)
        if sweep:
            res.extras["d2h_bytes"] += B * _lib.SWEEP_DTYPE.itemsize
        if field_cover:
            res.extras["d2h_bytes"] += B * _lib.PATH_COVER_DTYPE.itemsize
        if self.shard is not None:
            records = pf.hwin[:F * k * rec].view(_lib.SUMMARY_DTYPE).reshape(F, k)
            res.extras["winner_summary"] = records[:, 0].copy()
            res.extras["shard"] = self.shard
            res.extras["d2h_bytes"] += F * k * rec + 16
            if ranked:
                res.topk_summary = records
        elif ranked and len(res.summary) == B:
            res.topk_summary = np.zeros((F, k), dtype=_lib.SUMMARY_DTYPE)
            own = res.topk_cand >= 0
            res.topk_summary[own] = res.summary[res.topk_cand[own] - cand_base]
        res.extras["speculative"] = bool(buffers.speculative)
        if winners:
            # on the side stream: behind this batch (its event has completed), not behind later batches in flight
            with torch.cuda.stream(_side_stream(db.dev)):
                res.extras["d2h_bytes"] += fetch_winner_paths(db, res, outputs, slot=db.slot + 1)
        self._res = res
        return res


def run_device_batch(db: DeviceBatch, outputs: str = "summary", want_curvature: bool = False,
                     cost: str = "length", cand_base: int = 0, copy_summary: bool = True,
                     buffers: Optional[BatchBuffers] = None, fetch: bool = True,
                     winners: bool = False, corner_bits: bool = False, speculate: bool = False, wait: bool = True,
                     shard: Optional[tuple] = None, select: Optional[Selection] = None, obstacle_sweep: bool = False,
                     field_coverage: bool = False):
    """Enqueue one batch on torch's current stream and (``fetch``) copy summaries + the per-field best back.

    With ``buffers`` (from a previous run of the same batch shape) and ``db.max_points`` known the
    whole step is asynchronous: layout, prefix sum, plan, coverage and ranking kernels only.
    ``winners``: also bring every field's winning path and speeds to the host (``fetch_winner_paths``).
    ``speculate``: size the launch from remembered batches of the same shape instead of a synchronous layout
    read-back (``_Hints``; checked and repeated when the sizes do not fit).  ``wait=False`` returns a
    ``PendingBatch``.  ``shard=(lo, hi)``: the batch is this rank's candidates [lo, hi) of a batch sharded over the
    default process group; before the read-back the per-field ranking is merged over the ranks and the summary
    record of every ranked candidate gathered (``dist.reduce_topk``, ``dist.gather_winner_records``).  ``select``:
    the per-field top-k ranking (``BatchResult.topk_*``) instead of the argmin of ``cost``.  ``obstacle_sweep``: also
    each candidate's segment-level obstacle sweep (``BatchResult.sweep``; in a sharded batch, of this rank's
    candidates).  ``field_coverage`` (``outputs='paths'``): each candidate's whole-field and headland-band coverage
    (``BatchResult.field_cover``, likewise of this rank's candidates)."""
    if field_coverage and outputs != "paths":
        raise ValueError("field_coverage=True needs outputs='paths': it measures the materialised paths")
    if select is not None:
        selection = select
    else:   # the argmin of the length or of the time: the plain selections (include/fcpp.h)
        selection = Selection() if cost == "length" else Selection(w_length=0.0, w_time=1.0)
    return _run_device_batch(db, outputs, want_curvature, selection, select is not None, cand_base, copy_summary,
                             buffers, fetch, winners, corner_bits, speculate, wait, shard, obstacle_sweep, field_coverage)


def _run_device_batch(db: DeviceBatch, outputs: str, want_curvature: bool, selection: Selection, ranked: bool,
                      cand_base: int, copy_summary: bool, buffers: Optional[BatchBuffers], fetch: bool, winners: bool,
                      corner_bits: bool, speculate: bool, wait: bool, shard: Optional[tuple], obstacle_sweep: bool,
                      field_coverage: bool = False):
    """``run_device_batch`` with the ranking resolved: ``selection`` ranks every field, ``ranked`` = the caller asked
    for the ranking (``BatchResult.topk_*``)."""
    buffers, offsets = _launch_device_batch(db, outputs, want_curvature, selection, cand_base, buffers,
                                            corner_bits=corner_bits, speculate=speculate and copy_summary,
                                            sweep=obstacle_sweep, field_cover=field_coverage)
    if not fetch:
        return None
    win = None
    if shard is not None:
        from . import dist
        k = selection.top_k
        nfk = db.pb.n_fields * k
        dist.reduce_topk(buffers.d_cost[:nfk], buffers.d_best[:nfk], k)     # in place: the GLOBAL ranking
        # every rank passes the mask whether or not IT speculated: the all-reduce must have the same shape everywhere
        win = dist.gather_winner_records(buffers.d_sum, buffers.d_best[:nfk], shard[0], shard[1],
                                         count_mask=_SIZE_FLAGS)
    pf = _enqueue_fetch(db, buffers, outputs, offsets, copy_summary, cand_base, win, obstacle_sweep, field_coverage)
    pend = PendingBatch(db, pf, outputs, want_curvature, selection, ranked, cand_base, copy_summary, winners,
                        corner_bits, speculate and copy_summary, shard, obstacle_sweep, field_coverage)
    return pend if not wait else pend.result()


def plan_batch(fields, vehicle: Optional[VehicleParams] = None, candidates: Optional[Dict[str, np.ndarray]] = None,
               obstacles=None, start_points=None, outputs: str = "summary", grid_h: float = 0.1,
               coverage: bool = True, cost: str = "length", device=None, want_curvature: bool = False,
               distributed: bool = False, turn_model: str = "arc", clothoid_share: float = 0.5,
               winners: bool = False, wait: bool = True, select: Optional[Selection] = None,
               obstacle_sweep: bool = False, field_coverage: bool = False):
    """Evaluate B candidate plans.  See ``prepare_batch`` for the inputs.

    Returns a ``BatchResult``: per-candidate ``summary`` records (layout counts, path lengths and
    times per layer, accel/boundary/obstacle violation counts, headland and corner coverage cell
    counts, status) and the per-field argmin of ``cost`` ('length' = len_main+len_head metres,
    'time' = time_main+time_head seconds; ties to the lowest candidate index).

    ``turn_model='clothoid'`` (opt-in, SURVEY.md row A16) replaces the sampled circular arcs of the
    U-turns and headland corners by clothoid -> arc -> clothoid turns (same sample counts) whose
    Fresnel integrals are evaluated per sample point on the device; ``clothoid_share`` in (0, 1] is
    the share of each turn's deflection spent on the clothoids.

    ``turn_model='omega'`` (opt-in, the "Ω型跨行" pattern the reference only names, mlp3:312-320; build-defined and
    parity-unpinned like the clothoid): the rows of the main work are visited in skip order (blocks of 2 s rows,
    s = ceil(2 R / W), lower and upper half alternating) and every 20-sample turn connects the two swath ends — a
    half circle of radius gap / 2, or the Ω (bulb) turn of three radius-R arcs where the gap is below 2 R.  Rows,
    swath ends, sample counts and the headland are the U pattern's.

    ``winners=True`` also returns every field's winning path and speed profile on the host
    (``BatchResult.winner_paths``) — what a search caller needs from a batch.

    ``select=Selection(...)`` ranks each field's candidates under a weighted cost among those that respect the
    selection's limits (see ``Selection``) instead of the plain argmin: ``BatchResult.topk_cand`` / ``topk_cost`` /
    ``topk_summary`` hold the ``top_k`` best per field, ``best_cand`` / ``best_cost`` (and ``winners``) the first.
    It replaces ``cost``, which must stay 'length'.

    ``obstacle_sweep=True`` also measures how far each plan drives through the obstacles (DESIGN.md §3.9): D3's
    ``n_obstacle_viol`` counts path POINTS in the W/2-buffered obstacles, and a swath's two points can lie on either
    side of an obstacle; the sweep measures every SEGMENT.  ``BatchResult.sweep`` [B] (``_lib.SWEEP_DTYPE``) holds per
    layer the segments with metres inside the obstacle region and the sum of those metres.  It is read back with the
    summaries (no extra synchronisation) and changes no other output.

    ``field_coverage=True`` (needs ``outputs='paths'``) also measures how much of each field its plan covers
    (DESIGN.md §3.10): ``BatchResult.field_cover`` [B] (``_lib.PATH_COVER_DTYPE``) holds the cells of the whole field
    covered by the W/2 buffer of both layers, the headland band's cells covered by the headland layer (the
    summary's ``cov_total`` / ``cov_cells``) and D3's point counts, as ``verify_paths`` measures them on the same
    path.  Read back with the summaries; no other output changes.

    ``wait=False`` returns a ``PendingBatch`` as soon as the batch is enqueued; its ``result()`` gives the
    BatchResult.  Submitting the next batch before collecting the previous one overlaps the host side of a call with
    the kernels of the other (see ``PendingBatch``).

    ``distributed=True`` (inside a torch.distributed job): the candidates are sharded over the
    ranks in contiguous ranges, each rank plans its shard on its own GPU and the per-field best
    is merged with ONE all-gather of the (cost, candidate) words + a merge kernel (see ``dist.py``);
    ``winner_paths`` then holds the fields whose winner this rank owns."""
    if cost not in ("length", "time"):
        raise ValueError(f"cost must be 'length' or 'time', not {cost!r}")
    if field_coverage and outputs != "paths":
        raise ValueError("field_coverage=True needs outputs='paths': it measures the materialised paths")
    if select is not None:
        if not isinstance(select, Selection):
            raise ValueError(f"select must be a Selection, not {type(select).__name__}")
        select.check_batch(coverage, cost)
    vehicle = vehicle or VehicleParams()
    if distributed:
        from . import dist
        return dist.plan_batch_sharded(fields, vehicle, candidates, obstacles, start_points, outputs, grid_h,
                                       coverage, cost, device, want_curvature, turn_model, clothoid_share, winners, wait,
                                       select, obstacle_sweep, field_coverage)
    dev = _dev(device)
    pb = prepare_batch(fields, vehicle, candidates, obstacles, start_points, grid_h, coverage, turn_model,
                       clothoid_share)
    db = DeviceBatch(pb, dev)
    return run_device_batch(db, outputs, want_curvature, cost, winners=winners, speculate=True, wait=wait,
                            select=select, obstacle_sweep=obstacle_sweep, field_coverage=field_coverage)


def obstacle_sweep(paths, obstacles, working_width: float, n_main=None, device=None) -> np.ndarray:
    """The segment-level obstacle sweep of caller-supplied paths (DESIGN.md §3.9) on the GPU.

    ``paths``: one [n, 2] array or a sequence of them; ``obstacles``: one list of polygons (each a sequence of (x, y))
    that every path is checked against; the radius is ``working_width / 2``.  ``n_main`` (an int per path, or one int
    for a single path) splits a path into main work (its first n_main points) and headland, as a plan's
    ``main_work.path`` + ``headland.path``; without it the whole path counts as main work.  Returns a [n_paths]
    ``_lib.SWEEP_DTYPE`` array: per layer the segments that enter the obstacle region and the metres inside."""
    single = isinstance(paths, np.ndarray) and paths.ndim == 2
    plist = [paths] if single else list(paths)
    pts = [np.ascontiguousarray(np.asarray(p, dtype=np.float64).reshape(-1, 2)) for p in plist]
    n = len(pts)
    if n_main is not None:
        nm = np.atleast_1d(np.asarray(n_main, dtype=np.int64))
        if len(nm) != n:
            raise ValueError("n_main needs one value per path")
        if any(not 0 <= int(m) <= len(p) for m, p in zip(nm, pts)):
            raise ValueError("n_main must lie in [0, len(path)]")
        nm = nm.astype(np.int32)
    if not working_width > 0:
        raise ValueError("working_width must be > 0")
    polys = [np.asarray(o, dtype=np.float64).reshape(-1, 2) for o in (obstacles or []) if len(o)]
    out = np.zeros(n, dtype=_lib.SWEEP_DTYPE)
    if n == 0:
        return out
    dev = _dev(device)
    h = _lib.handle(dev.index)
    offs = np.zeros(n + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(p) for p in pts])
    arrays = {"path": np.concatenate(pts) if offs[-1] else np.zeros((1, 2)), "offsets": offs,
              "vs": np.concatenate([[0], np.cumsum([len(o) for o in polys])]).astype(np.int32),
              "verts": np.concatenate(polys) if polys else np.zeros((1, 2))}
    if n_main is not None:
        arrays["n_main"] = nm
    with torch.cuda.device(dev):
        t = _pack_to_dev(arrays, dev)
        d_out = torch.empty(n * _lib.SWEEP_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        h.check(h.lib.fcpp_obstacle_sweep_paths(h.h, t["path"].data_ptr(), t["offsets"].data_ptr(), n,
                                                t["n_main"].data_ptr() if n_main is not None else None,
                                                t["vs"].data_ptr(), t["verts"].data_ptr(), len(polys),
                                                float(working_width) / 2, d_out.data_ptr(), stream))
        out[:] = d_out.cpu().numpy().view(_lib.SWEEP_DTYPE)
    return out



def _fields_array(fields) -> np.ndarray:
    fv = np.asarray(fields, dtype=np.float64)
    if fv.shape == (4, 2):
        fv = fv[None]
    if fv.ndim != 3 or fv.shape[1:] != (4, 2) or len(fv) == 0:
        raise ValueError("fields must be one [4, 2] quad or an [F, 4, 2] array of them")
    if not np.isfinite(fv).all():
        raise ValueError("field vertices must be finite")
    e = np.roll(fv, -1, axis=1) - fv
    cross = e[:, :, 0] * np.roll(e, -1, axis=1)[:, :, 1] - e[:, :, 1] * np.roll(e, -1, axis=1)[:, :, 0]
    if not (cross > 0).all():
        raise ValueError("every field must be a convex counter-clockwise quad")
    return np.ascontiguousarray(fv)


def _per_path(v, n: int, name: str, dtype) -> np.ndarray:
    a = np.asarray(v, dtype=dtype)
    if a.ndim == 0:
        a = np.full(n, a, dtype=dtype)
    if a.shape != (n,):
        raise ValueError(f"{name} needs one value per path ({n}), not shape {a.shape}")
    return np.ascontiguousarray(a)


def verify_paths(paths, fields, vehicle: Optional[VehicleParams] = None, *, path_field=None, headland_width=None,
                 obstacles=None, n_main=None, grid_h: float = 0.1, device=None) -> np.ndarray:
    """The checks every generated plan carries, for caller-supplied paths on the GPU (DESIGN.md §3.10).

    ``paths``: one [n, 2] array or a sequence of them (any lengths, 0 and 1 points too); ``fields``: one [4, 2] convex
    CCW quad or [F, 4, 2] of them; ``path_field``: each path's field (may be omitted with one field);
    ``headland_width`` (one value or one per path; default ``vehicle.min_turn_radius``): the band's R;
    ``obstacles``: one (possibly empty) polygon list per field, as ``plan_batch``; the radius is
    ``vehicle.working_width / 2``.  ``n_main`` (one int per path, or one int for a single path) splits a path into main
    work (its first n_main points) and headland.  Without it n_main = 0: the whole path is the HEADLAND layer and counts
    for both the band and the field (unlike ``obstacle_sweep``, whose default is all main work).

    Returns a [n_paths] ``_lib.PATH_COVER_DTYPE`` array: D3's ``n_boundary_viol`` / ``n_obstacle_viol`` over every
    point; ``band_total`` / ``band_cells``, the A11 headland band of (field, headland width) and its cells covered by
    the headland layer (a plan's ``cov_total`` / ``cov_cells``); ``field_total`` / ``field_cells``, the whole field's
    cells and those covered by both layers (the segment joining the layers counts for neither).  ``status``
    ``_lib.PATH_OUT_OF_RANGE``: a point lies ~107 km or more from its field (every count 0).  Every input is checked
    on the host before the device is touched: invalid input raises ValueError."""
    vehicle = vehicle or VehicleParams()
    fv = _fields_array(fields)
    F = len(fv)
    single = isinstance(paths, np.ndarray) and paths.ndim == 2
    plist = [paths] if single else list(paths)
    pts = []
    for p in plist:
        a = np.asarray(p, dtype=np.float64)
        if a.size == 0:
            a = a.reshape(0, 2)
        if a.ndim != 2 or a.shape[1] != 2:
            raise ValueError(f"every path must be an [n, 2] array, not shape {a.shape}")
        if not np.isfinite(a).all():
            raise ValueError("path coordinates must be finite")
        pts.append(np.ascontiguousarray(a))
    n = len(pts)
    lens = np.array([len(p) for p in pts], dtype=np.int64)
    if path_field is None:
        if F != 1:
            raise ValueError("path_field is required with more than one field")
        path_field = 0
    pf = _per_path(path_field, n, "path_field", np.int64)
    if n and (pf.min() < 0 or pf.max() >= F):
        raise ValueError(f"path_field must lie in [0, {F})")
    hw = _per_path(vehicle.min_turn_radius if headland_width is None else headland_width, n, "headland_width",
                   np.float64)
    if not np.isfinite(hw).all():
        raise ValueError("headland_width must be finite")
    nm = np.zeros(n, dtype=np.int64)
    if n_main is not None:
        nm = np.atleast_1d(np.asarray(n_main))
        if nm.ndim != 1 or len(nm) != n or not np.issubdtype(nm.dtype, np.integer):
            raise ValueError("n_main needs one integer per path")
        nm = nm.astype(np.int64)
        if ((nm < 0) | (nm > lens)).any():
            raise ValueError("n_main must lie in [0, len(path)]")
    W = float(vehicle.working_width)
    if not (W > 0 and math.isfinite(W)):
        raise ValueError("working_width must be > 0")
    hq = float(grid_h) * 1e4
    if not (grid_h > 0 and math.isfinite(hq) and abs(hq - round(hq)) <= 1e-6 and round(hq) % 2 == 0):
        raise ValueError(f"grid_h must be a positive even multiple of 1e-4 m, not {grid_h!r}")
    if obstacles is not None:
        for polys in obstacles:
            for poly in polys:
                o = np.asarray(poly, dtype=np.float64)
                if o.ndim != 2 or o.shape[1] != 2 or len(o) < 3 or not np.isfinite(o).all():
                    raise ValueError("every obstacle must be a polygon of >= 3 finite (x, y) vertices")
    arrays: Dict[str, np.ndarray] = {}
    _obstacle_tables(obstacles, F, W, arrays)
    out = np.zeros(n, dtype=_lib.PATH_COVER_DTYPE)
    if n == 0:
        return out
    offs = np.zeros(n + 1, dtype=np.int64)
    offs[1:] = np.cumsum(lens)
    arrays.update({"path": np.concatenate(pts) if offs[-1] else np.zeros((1, 2)), "offsets": offs,
                   "field": pf.astype(np.int32), "hw": hw, "n_main": nm.astype(np.int32), "field_verts": fv})
    dev = _dev(device)
    h = _lib.handle(dev.index)
    with torch.cuda.device(dev):
        t = _pack_to_dev(arrays, dev)
        d_out = torch.empty(n * _lib.PATH_COVER_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        obs = t.get("obs_poly_start")
        h.check(h.lib.fcpp_path_coverage(h.h, t["path"].data_ptr(), t["offsets"].data_ptr(), n, t["n_main"].data_ptr(),
                                         t["field"].data_ptr(), t["hw"].data_ptr(), F, t["field_verts"].data_ptr(),
                                         obs.data_ptr() if obs is not None else None,
                                         t["obs_vert_start"].data_ptr() if obs is not None else None,
                                         t["obs_verts"].data_ptr() if obs is not None else None, W / 2, float(grid_h),
                                         d_out.data_ptr(), stream))
        out[:] = d_out.cpu().numpy().view(_lib.PATH_COVER_DTYPE)
    return out
