"""Drop-in for the reference's single-field planner class (SURVEY.md §8(b)).

``TwoLayerPathPlannerV37`` mirrors ``multi_layer_planner_v3.TwoLayerPathPlannerV37`` (mlp3:42):
same constructor keywords, same attributes, same result dict, same ``verify_*`` methods — but
every compute step runs in the CUDA library (a batch of ONE candidate through the same kernels
that ``plan_batch`` uses).  The reference prints ~60 lines per plan; here output is opt-in
(``verbose=True`` prints a short summary) because prints are not part of the result contract.

Aliases that callers of the reference expect (SURVEY.md F2/F3): ``TwoLayerPathPlannerV35``,
``TwoLayerPathPlannerV36`` (test scripts, multi_field_planner.py:24), and the README names
``TwoLayerPlannerV35`` / ``TwoLayerPlannerV36`` which take ``vehicle=`` and expose ``.plan()``
(README.md:257-285).
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _geometry as G
from . import _lib
from .batch import DeviceBatch, _dev, corner_grids, obstacle_sweep, prepare_batch, run_device_batch, verify_paths
from .vehicle import VehicleParams

APPROACH_POINTS = 50  # mlp3:1317
GRID_RESOLUTION = 0.1  # mlp3:1452


class TwoLayerPathPlannerV37:
    def __init__(self, vehicle_params: VehicleParams = None, field_length: float = None,
                 field_width: float = None, field_vertices: List[Tuple[float, float]] = None,
                 obstacles: List[List[Tuple[float, float]]] = None, start_point: Tuple[float, float] = None,
                 end_point: Tuple[float, float] = None, *, vehicle: VehicleParams = None, device=None,
                 verbose: bool = False, grid_h: float = 0.1, turn_model: str = "arc", clothoid_share: float = 0.5):
        if vehicle_params is None:
            vehicle_params = vehicle          # README spelling (README.md:262-266)
        if vehicle_params is None:
            vehicle_params = VehicleParams()
        self.vehicle = vehicle_params
        self.obstacles = obstacles or []
        self.verbose = verbose
        self.grid_h = grid_h
        self.turn_model = turn_model          # 'arc' = reference behaviour; 'clothoid' = opt-in (README.md:105-113)
        self.clothoid_share = clothoid_share
        self._device = device
        self._process_field_input(field_length, field_width, field_vertices)
        self.corner_angles = [float(a) for a in G.corner_angles_deg(np.asarray(self.field_vertices, dtype=np.float64)[None])[0]] \
            if len(self.field_vertices) == 4 else []
        self.field_shape = self._detect_field_shape()
        self.headland_width = self.vehicle.min_turn_radius          # mlp3:295-310
        self.main_work_pattern = self._select_main_work_pattern()
        self.start_point = self._validate_point(start_point)
        self.end_point = self._validate_point(end_point)
        self._last = None
        self._last_path = None     # (points [n, 2], n_main) of the last plan
        self._last_grids = None

    # ---- A2: field set-up (host, FP64) -----------------------------------------------------
    def _process_field_input(self, field_length, field_width, field_vertices):
        """mlp3:109-135."""
        if field_vertices is not None:
            self.field_vertices = [tuple(v) for v in field_vertices]
            v = np.asarray(self.field_vertices, dtype=np.float64)
            self.field_length = float(v[:, 0].max() - v[:, 0].min())
            self.field_width = float(v[:, 1].max() - v[:, 1].min())
        elif field_length is not None and field_width is not None:
            self.field_length = field_length
            self.field_width = field_width
            self.field_vertices = [(0, 0), (field_length, 0), (field_length, field_width), (0, field_width)]
        else:
            raise ValueError("必须提供 field_vertices 或 (field_length, field_width)")
        self.field_polygon = G.QuadPolygon(self.field_vertices)

    def _calculate_corner_angle(self, corner_index: int) -> float:
        return self.corner_angles[corner_index]

    def _detect_field_shape(self) -> str:
        """mlp3:137-163, :194-222."""
        if len(self.field_vertices) != 4:
            return 'other'
        if all(abs(a - 90) < 1.0 for a in self.corner_angles):
            return 'rectangle'
        v = np.asarray(self.field_vertices, dtype=np.float64)
        e = np.roll(v, -1, axis=0) - v

        def par(a, b, tol=0.01):
            return abs(a[0] * b[1] - a[1] * b[0]) < tol * (np.linalg.norm(a) * np.linalg.norm(b))

        return 'parallelogram' if par(e[0], e[2]) and par(e[1], e[3]) else 'other'

    def _select_main_work_pattern(self) -> str:
        """mlp3:312-320 (a label only, SURVEY.md F4)."""
        return "Ω型跨行" if self.field_length / self.field_width < 1.5 else "U型往复"

    def _validate_point(self, point):
        """mlp3:322-343 — closed test against the bbox EXTENTS anchored at the origin (Q11)."""
        if point is None:
            return None
        x, y = point
        if not (0 <= x <= self.field_length and 0 <= y <= self.field_width):
            return None
        return (x, y)

    def _get_possible_start_corners(self):
        w = self.headland_width
        return [(w / 2, w / 2, "左下角"), (self.field_length - w / 2, w / 2, "右下角"),
                (self.field_length - w / 2, self.field_width - w / 2, "右上角"),
                (w / 2, self.field_width - w / 2, "左上角")]

    def _select_best_start_corner(self, parking_position):
        """mlp3:360-385 — first minimum wins."""
        cs = self._get_possible_start_corners()
        d = [float(np.sqrt((x - parking_position[0]) ** 2 + (y - parking_position[1]) ** 2)) for x, y, _ in cs]
        i = int(min(range(4), key=lambda k: d[k]))
        return i, (cs[i][0], cs[i][1]), cs[i][2]

    # ---- the plan ---------------------------------------------------------------------------
    def _require_quad(self):
        if len(self.field_vertices) != 4:
            raise ValueError("only 4-vertex fields are supported (the reference's corner logic, mlp3:983-1007)")
        if G.shoelace(self.field_vertices) <= 0:
            raise ValueError("field_vertices must be counter-clockwise (vertex 0 = lower-left, mlp3:127-132)")

    def plan_complete_coverage(self) -> Dict:
        """mlp3:387-465: start corner -> layer 1 -> layer 2 -> speed planning on the concatenation
        -> per-layer stats -> approach/departure lines -> result dict."""
        t0 = time.time()
        self._require_quad()
        sci = 0
        if self.start_point:
            sci, _, _ = self._select_best_start_corner(self.start_point)
        cands = {"field_id": np.zeros(1, dtype=np.int32), "start_corner": np.array([sci], dtype=np.int32)}
        sp = np.array([[np.nan, np.nan]]) if not self.start_point else np.array([self.start_point], dtype=np.float64)
        pb = prepare_batch([self.field_vertices], self.vehicle, cands, [self.obstacles], sp, self.grid_h, True,
                           self.turn_model, self.clothoid_share)
        # start_corner only selects the headland start; the pass order comes from the start point
        # (mlp3:649-658) or stays (False, False) without one
        if not self.start_point:
            pb.arrays["cand_flags"] &= ~np.int32(_lib.FLAG_REVERSE_ORDER | _lib.FLAG_START_FROM_RIGHT)
        db = DeviceBatch(pb, _dev(self._device), pin=False)
        res = run_device_batch(db, outputs="paths", corner_bits=True)
        s = res.summary[0]
        if s["status"] & _lib.CAND_INSET_EMPTY:
            raise ValueError(f"田头宽度{self.headland_width}m过大，无法定义主作业区域")  # mlp3:598
        if s["status"] & _lib.CAND_LOOP_SKIPPED:
            raise ValueError("all the input array dimensions except for the concatenation axis must match "
                             "exactly (headland loop skipped, mlp3:967-969 + :939)")
        if s["status"]:
            raise _lib.FcppError(f"plan failed with candidate status {int(s['status'])}")
        path, speeds, nm = res.path(0)
        main_inset = G.mitred_inset(self.field_vertices, self.headland_width)
        holes = [G.round_buffer_moments(o, self.vehicle.working_width / 2) for o in self.obstacles]
        main_area = G.QuadPolygon(main_inset, holes)
        head_area = G.QuadPolygon(self.field_vertices, inner=G.QuadPolygon(main_inset))
        lm, lh = float(s["len_main"]), float(s["len_head"])
        main = {'path': path[:nm].copy(), 'speeds': speeds[:nm].copy(), 'pattern': self.main_work_pattern,
                'area': main_area,
                'stats': {'path_length_km': lm / 1000, 'time_hours': float(s["time_main"]) / 3600,
                          # stale on purpose: computed from the PRE-adjustment speeds (Q8, mlp3:616-628)
                          'avg_speed_kmh': (lm / 1000) / (float(s["time_main_pre"]) / 3600)
                          if s["time_main_pre"] > 0 else 0}}
        head = {'path': path[nm:].copy(), 'speeds': speeds[nm:].copy(), 'area': head_area,
                'stats': {'path_length_km': lh / 1000, 'time_hours': float(s["time_head"]) / 3600,
                          'avg_speed_kmh': (lh / 1000) / (float(s["time_head_pre"]) / 3600)
                          if s["time_head_pre"] > 0 else 0,
                          # integer raster of the headland band (D5) instead of GEOS areas
                          'coverage_rate': (int(s["cov_cells"]) / int(s["cov_total"])) if s["cov_total"] else 0.0}}
        approach = departure = None
        if self.start_point:   # mlp3:437-441: targets headland.path[0] (Q12)
            approach = self._generate_approach_path(self.start_point, head['path'][0])
        if self.end_point:     # mlp3:443-447
            departure = self._generate_departure_path(head['path'][-1], self.end_point)
        self._last = s
        self._last_path = (path, nm)
        self._last_grids = corner_grids(res.extras["corner_bits"][0].cpu().numpy().view(np.uint32), int(s["corner_g"])) \
            if not (s["status"] & _lib.CAND_GRID_TOO_LARGE) else None
        result = {'main_work': main, 'headland': head, 'approach_path': approach, 'departure_path': departure,
                  'total_time': time.time() - t0, 'version': 'V3.5.1',
                  'features': ['真正两层', '切线倒车', '网格验证', '强制降速', '智能起点'],
                  # extension (not in the reference dict): the validation summary of this plan
                  'validation': {k: (s[k].tolist() if hasattr(s[k], "tolist") else s[k]) for k in s.dtype.names}}
        if self.verbose:
            print(f"[fcpp] plan: main {nm} pts {lm/1000:.3f} km, headland {len(path)-nm} pts {lh/1000:.3f} km, "
                  f"{result['total_time']*1e3:.1f} ms")
        return result

    plan = plan_complete_coverage   # README.md:272

    # ---- A14 (host, 50-point lines) --------------------------------------------------------------
    def _generate_approach_path(self, start, end, num_points: int = APPROACH_POINTS) -> np.ndarray:
        """mlp3:1313-1333."""
        return np.column_stack([np.linspace(start[0], end[0], num_points), np.linspace(start[1], end[1], num_points)])

    _generate_departure_path = _generate_approach_path   # mlp3:1335-1355

    # ---- device-backed helpers on caller-supplied paths ------------------------------------------
    def _speed_verify(self, path, speeds, do_speed_plan: bool):
        dev = _dev(self._device)
        h = _lib.handle(dev.index)
        path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 2)
        n = len(path)
        speeds = np.ascontiguousarray(speeds if speeds is not None else np.zeros(n), dtype=np.float64)
        v = self.vehicle
        veh = _lib.Vehicle(v.working_width, v.max_work_speed_kmh, v.max_headland_speed_kmh, v.headland_turn_speed_kmh,
                           v.max_lateral_accel, v.max_longitudinal_accel, v.safety_factor, 2.5)
        with torch.cuda.device(dev):
            d_p = torch.from_numpy(path).to(dev)
            d_s = torch.from_numpy(speeds).to(dev)
            d_o = torch.tensor([0, n], dtype=torch.int64, device=dev)
            d_out = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
            d_sum = torch.zeros(_lib.SUMMARY_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            h.check(h.lib.fcpp_speed_verify(h.h, C.byref(veh), d_p.data_ptr(), d_s.data_ptr(), d_o.data_ptr(), 1, n,
                                            1 if do_speed_plan else 0, d_out.data_ptr(), None, d_sum.data_ptr(), st))
            s = d_sum.cpu().numpy().view(_lib.SUMMARY_DTYPE)[0]
            out = d_out.cpu().numpy()[:n]
        if s["status"] & _lib.CAND_TOO_LARGE:
            raise _lib.FcppError(f"path of {n} points exceeds the on-chip staging capacity")
        return s, out

    def _apply_curvature_based_speed_limit(self, path, speeds) -> np.ndarray:
        """mlp3:467-511 on a caller-supplied path."""
        if len(path) < 3:
            return speeds
        return self._speed_verify(path, speeds, True)[1]

    def _calculate_path_length(self, path) -> float:
        """mlp3:1290-1296 (called by test/test_v351_start_end_points.py:133)."""
        if len(path) < 2:
            return 0.0
        return float(self._speed_verify(path, None, False)[0]["len_main"])

    def _calculate_work_time(self, path, speeds) -> float:
        """mlp3:1298-1311."""
        if len(path) < 2 or len(speeds) == 0:
            return 0.0
        return float(self._speed_verify(path, speeds, False)[0]["time_main"])

    def verify_curvature_constraints(self, path, speeds) -> Dict:
        """mlp3:1373-1424."""
        if len(path) < 3:
            return {'max_curvature': 0, 'violations': 0, 'pass': True}
        s, _ = self._speed_verify(path, speeds, False)
        n = len(path) - 2
        viol = int(s["n_accel_viol"])
        rate = viol / n * 100 if n > 0 else 0
        return {'max_curvature': float(s["max_curvature"]), 'max_lateral_accel': float(s["max_lateral_accel"]),
                'max_allowed_accel': self.vehicle.max_lateral_accel, 'accel_violations': viol,
                'accel_violation_rate': rate, 'max_jump': float(s["max_jump"]), 'pass': rate < 5}

    def verify_obstacle_clearance(self, path=None, n_main: Optional[int] = None) -> Dict:
        """How far a path drives through the obstacles buffered by W/2 (the segment-level sweep, DESIGN.md §3.9).

        ``path=None``: the last plan (``main_work.path`` then ``headland.path``, planned first if there is none);
        otherwise a caller-supplied [n, 2] path whose first ``n_main`` points are main work (default: all of them).
        Returns per layer the segments that enter the obstacle region and the metres inside, their totals,
        ``pass`` = no segment enters, and ``point_violations``: D3's count of path POINTS inside (the plan's
        ``n_obstacle_viol``; None for a caller-supplied path) — a swath can cross an obstacle with both its points
        outside, which the point count does not see."""
        points = None
        if path is None:
            if self._last_path is None:
                self.plan_complete_coverage()
            path, n_main = self._last_path
            points = int(self._last["n_obstacle_viol"])
        path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 2)
        sw = obstacle_sweep(path, self.obstacles, self.vehicle.working_width,
                            n_main=None if n_main is None else [int(n_main)], device=self._device)[0]
        segs = int(sw["n_seg_main"]) + int(sw["n_seg_head"])
        return {'segments_main': int(sw["n_seg_main"]), 'segments_head': int(sw["n_seg_head"]),
                'metres_main': float(sw["len_main"]), 'metres_head': float(sw["len_head"]),
                'segments': segs, 'metres': float(sw["len_main"]) + float(sw["len_head"]),
                'point_violations': points, 'pass': segs == 0}

    def verify_field_coverage(self, path=None, n_main: Optional[int] = None) -> Dict:
        """How much of the field a path covers, on the A11 lattice (DESIGN.md §3.10).

        ``path=None``: the last plan (``main_work.path`` then ``headland.path``, planned first if there is none);
        otherwise a caller-supplied [n, 2] path whose first ``n_main`` points are main work — without ``n_main`` the
        whole path is the headland layer (unlike ``verify_obstacle_clearance``, whose default is all main work).
        Returns ``field_coverage_rate`` (cells of the whole field covered by the W/2 buffer of both layers),
        ``band_coverage_rate`` (the headland band's cells covered by the headland layer: the plan's ``coverage_rate``),
        their cells and totals, and D3's point counts ``boundary_violations`` / ``obstacle_violations``."""
        if path is None:
            if self._last_path is None:
                self.plan_complete_coverage()
            path, n_main = self._last_path
        path = np.ascontiguousarray(path, dtype=np.float64).reshape(-1, 2)
        r = verify_paths([path], [self.field_vertices], self.vehicle, headland_width=self.headland_width,
                         obstacles=[self.obstacles], n_main=[0 if n_main is None else int(n_main)], grid_h=self.grid_h,
                         device=self._device)[0]
        ft, fc, bt, bc = (int(r[k]) for k in ("field_total", "field_cells", "band_total", "band_cells"))
        return {'field_coverage_rate': fc / ft if ft else 0.0, 'band_coverage_rate': bc / bt if bt else 0.0,
                'field_cells': fc, 'field_total': ft, 'band_cells': bc, 'band_total': bt,
                'boundary_violations': int(r["n_boundary_viol"]), 'obstacle_violations': int(r["n_obstacle_viol"]),
                'status': int(r["status"])}

    def verify_corner_coverage_grid_based(self, corner, corner_index: int, turn_path, reverse_path=None) -> Dict:
        """mlp3:1426-1510 with the exact fixed-point predicate (D5)."""
        R, W = self.vehicle.min_turn_radius, self.vehicle.working_width
        g = int(2 * R / GRID_RESOLUTION)                                   # mlp3:1457
        x, y = corner
        ox = x if corner_index in (0, 3) else x - 2 * R                    # mlp3:1461-1468
        oy = y if corner_index in (0, 1) else y - 2 * R
        # the window raster's range contract (include/fcpp.h fcpp_raster_window), checked before the device is touched
        o = np.rint(np.array([ox, oy], dtype=np.float64) * 1e4)
        for name, p in (("turn_path", turn_path), ("reverse_path", reverse_path)):
            if p is None or len(p) == 0:
                continue
            d = np.abs(np.rint(np.asarray(p, dtype=np.float64).reshape(-1, 2) * 1e4) - o)
            bad = np.nonzero(~(d < 2.0 ** 30).all(axis=1))[0]
            if len(bad):
                raise ValueError(f"{name} point {int(bad[0])} lies 2^30 lattice units (~107 km) or more from the "
                                 f"corner window's origin {(ox, oy)}")
        dev = _dev(self._device)
        h = _lib.handle(dev.index)
        nw = (g * g + 31) // 32
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            d_bits = torch.zeros(nw, dtype=torch.int32, device=dev)
            d_cnt = torch.zeros(1, dtype=torch.int64, device=dev)
            counts = []
            for p in (turn_path, reverse_path):
                if p is None or len(p) == 0:
                    counts.append(counts[-1] if counts else 0)
                    continue
                d_p = torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64).reshape(-1, 2)).to(dev)
                h.check(h.lib.fcpp_raster_window(h.h, d_p.data_ptr(), len(p), W / 2, ox, oy, GRID_RESOLUTION, g,
                                                 d_bits.data_ptr(), d_cnt.data_ptr(), st))
                counts.append(int(d_cnt.item()))
            words = d_bits.cpu().numpy().view(np.uint32)
        grid = np.unpackbits(words.view(np.uint8), bitorder="little")[:g * g].reshape(g, g).astype(bool)
        before = counts[0] / (g * g) * 100
        after = counts[1] / (g * g) * 100
        return {'coverage_before': before, 'coverage_after': after, 'improvement': after - before, 'grid': grid,
                'grid_origin': (ox, oy), 'grid_resolution': GRID_RESOLUTION,
                'cells_before': counts[0], 'cells_after': counts[1]}

    def verify_all_corners_coverage(self, headland_result: Dict = None) -> Dict:
        """mlp3:1512-1578: the four MAIN-AREA corners with freshly generated arcs (Q15); the counts
        come from the batched coverage kernel of the last plan (recomputed if there is none)."""
        if self._last is None:
            self.plan_complete_coverage()
        s = self._last
        g2 = float(int(s["corner_g"]) ** 2)
        R, hw = self.vehicle.min_turn_radius, self.headland_width
        # mlp3:1531-1536 corner positions and mlp3:1461-1468 window origins
        pos = [(hw, hw), (self.field_length - hw, hw), (self.field_length - hw, self.field_width - hw),
               (hw, self.field_width - hw)]
        corners = []
        for c in range(4):
            b, a = int(s["corner_before"][c]) / g2 * 100, int(s["corner_after"][c]) / g2 * 100
            x, y = pos[c]
            origin = (x if c in (0, 3) else x - 2 * R, y if c in (0, 1) else y - 2 * R)
            corners.append({'coverage_before': b, 'coverage_after': a, 'improvement': a - b,
                            # the occupancy grid after the reverse fill, grid[j, i] (mlp3:1477, :1503-1510): written
                            # out by the coverage kernel from its shared-memory tile
                            'grid': self._last_grids[c] if self._last_grids is not None else None,
                            'grid_origin': origin,
                            'cells_before': int(s["corner_before"][c]), 'cells_after': int(s["corner_after"][c]),
                            'grid_resolution': GRID_RESOLUTION})
        ab = float(np.mean([c['coverage_before'] for c in corners]))
        aa = float(np.mean([c['coverage_after'] for c in corners]))
        return {'corners': corners, 'avg_coverage_before': ab, 'avg_coverage_after': aa, 'avg_improvement': aa - ab}


# names other files of the reference import (SURVEY.md F2/F3)
TwoLayerPathPlannerV35 = TwoLayerPathPlannerV37
TwoLayerPathPlannerV36 = TwoLayerPathPlannerV37
TwoLayerPlannerV35 = TwoLayerPathPlannerV37
TwoLayerPlannerV36 = TwoLayerPathPlannerV37
TwoLayerPlannerV37 = TwoLayerPathPlannerV37
