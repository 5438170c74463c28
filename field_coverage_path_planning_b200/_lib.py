"""ctypes binding of libfcpp.so (the C-ABI declared in include/fcpp.h).

There is NO CPU fallback: if the shared library is missing or no CUDA device is usable, the
functions here raise — loudly — instead of computing anything on the host.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FCPP_LIB selects another build of the same library (A/B timing of kernel variants); there is still
# no fallback: the file must exist and export the ABI
LIB_PATH = os.environ.get("FCPP_LIB") or os.path.join(_HERE, "libfcpp.so")
ABI_VERSION = 5

FLAG_CORNER_MASK = 3
FLAG_REVERSE_ORDER = 4
FLAG_START_FROM_RIGHT = 8
FLAG_ROTATED = 16
FLAG_GAP_GATE = 32
FLAG_START_POINT = 64

CAND_INSET_EMPTY = 1
CAND_LOOP_SKIPPED = 2
CAND_TOO_MANY_LOOPS = 4
CAND_TOO_LARGE = 8
CAND_GRID_TOO_LARGE = 16


class FcppError(RuntimeError):
    pass


class Vehicle(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "working_width", "max_work_speed_kmh", "max_headland_speed_kmh", "headland_turn_speed_kmh",
        "max_lateral_accel", "max_longitudinal_accel", "safety_factor", "reverse_speed_kmh")]


class Batch(C.Structure):
    _fields_ = [
        ("vehicle", Vehicle),
        ("n_fields", C.c_int32),
        ("field_verts", C.c_void_p),
        ("field_extent", C.c_void_p),
        ("field_flags", C.c_void_p),
        ("obs_poly_start", C.c_void_p),
        ("obs_vert_start", C.c_void_p),
        ("obs_verts", C.c_void_p),
        ("obs_moments", C.c_void_p),
        ("max_obs_verts", C.c_int32),
        ("max_obs_polys", C.c_int32),
        ("n_cand", C.c_int64),
        ("cand_field", C.c_void_p),
        ("cand_R", C.c_void_p),
        ("cand_rot", C.c_void_p),
        ("cand_flags", C.c_void_p),
        ("cand_start", C.c_void_p),
        ("grid_h", C.c_double),
        ("do_coverage", C.c_int32),
        ("max_points_hint", C.c_int32),
        ("max_head_points_hint", C.c_int32),
        ("turn_model", C.c_int32),
        ("cover_dedupe", C.c_int32),
        ("clothoid_share", C.c_double),
        ("n_ax_headings", C.c_int32),
        ("n_ax_radii", C.c_int32),
        ("n_ax_corners", C.c_int32),
        ("ax_default_radius_flags", C.c_int32),
        ("ax_heading_rot", C.c_void_p),
        ("ax_heading_flags", C.c_void_p),
        ("ax_radii", C.c_void_p),
        ("ax_radius_flags", C.c_void_p),
        ("ax_corners", C.c_void_p),
        ("field_rot", C.c_void_p),
        ("field_rot_flags", C.c_void_p),
        ("ax_default_radius", C.c_double),
        ("cand_first", C.c_int64),
    ]


class Outputs(C.Structure):
    _fields_ = [
        ("summary", C.c_void_p),
        ("offsets", C.c_void_p),
        ("path_xy", C.c_void_p),
        ("speeds_kmh", C.c_void_p),
        ("curvature", C.c_void_p),
        ("path_capacity", C.c_int64),
        ("corner_bits", C.c_void_p),
        ("corner_bits_stride", C.c_int64),
    ]


class GAConfigC(C.Structure):
    """fcpp_ga_config (GAConfig ga:20-29 + seed)."""
    _fields_ = [
        ("population_size", C.c_int32), ("max_generations", C.c_int32),
        ("crossover_rate", C.c_double), ("mutation_rate", C.c_double),
        ("elite_size", C.c_int32), ("tournament_size", C.c_int32),
        ("convergence_threshold", C.c_int32), ("check_every", C.c_int32),
        ("seed", C.c_uint64),
    ]


class GAResultC(C.Structure):
    """fcpp_ga_result (stats of ga:122-127)."""
    _fields_ = [
        ("generations", C.c_int32), ("convergence_gen", C.c_int32), ("final_population", C.c_int32),
        ("reserved", C.c_int32), ("best_distance", C.c_double), ("best_fitness", C.c_double),
    ]


class SelectionC(C.Structure):
    """fcpp_selection (include/fcpp.h): weights, cell area, limits (< 0: none), top_k."""
    _fields_ = [(n, C.c_double) for n in (
        "w_length", "w_time", "w_boundary", "w_obstacle", "w_accel", "w_uncovered", "cell_area", "min_coverage")] + [
        (n, C.c_int32) for n in ("max_boundary_viol", "max_obstacle_viol", "max_accel_viol", "top_k")]


SELECT_MAX_K = 32
GA_TRACE_INTS = 48
GA_MAX_TOURNAMENT = 16

# numpy mirror of fcpp_summary (176 bytes)
SUMMARY_DTYPE = np.dtype([
    ("status", "<i4"), ("n_passes", "<i4"), ("n_loops", "<i4"), ("n_main", "<i4"), ("n_head", "<i4"),
    ("n_rev", "<i4", (3,)), ("n_accel_viol", "<i4"), ("n_boundary_viol", "<i4"), ("n_obstacle_viol", "<i4"),
    ("corner_g", "<i4"), ("corner_before", "<i4", (4,)), ("corner_after", "<i4", (4,)),
    ("cov_cells", "<i8"), ("cov_total", "<i8"),
    ("len_main", "<f8"), ("len_head", "<f8"), ("time_main", "<f8"), ("time_head", "<f8"),
    ("time_main_pre", "<f8"), ("time_head_pre", "<f8"),
    ("max_curvature", "<f8"), ("max_lateral_accel", "<f8"), ("max_jump", "<f8"), ("reserved", "<f8"),
], align=True)
assert SUMMARY_DTYPE.itemsize == 176, SUMMARY_DTYPE.itemsize

# numpy mirror of fcpp_sweep (24 bytes): per layer, the segments that enter the obstacle region and the metres inside
SWEEP_DTYPE = np.dtype([("n_seg_main", "<i4"), ("n_seg_head", "<i4"), ("len_main", "<f8"), ("len_head", "<f8")],
                       align=True)
assert SWEEP_DTYPE.itemsize == 24, SWEEP_DTYPE.itemsize

EXPORTS = [
    "fcpp_abi_version", "fcpp_create", "fcpp_destroy", "fcpp_last_error", "fcpp_set_trig_tables",
    "fcpp_layout", "fcpp_plan_batch", "fcpp_obstacle_sweep", "fcpp_obstacle_sweep_paths", "fcpp_field_select", "fcpp_field_select_merge", "fcpp_winner_records", "fcpp_status_count", "fcpp_speed_verify", "fcpp_raster_window",
    "fcpp_tour_lengths", "fcpp_distance_matrix", "fcpp_connection_matrix", "fcpp_ga_init_population", "fcpp_ga_next_size", "fcpp_ga_generation", "fcpp_ga_solve", "fcpp_kmeans_lloyd", "fcpp_tsp_two_opt",
    "fcpp_launch_count", "fcpp_last_max_points", "fcpp_last_max_head_points", "fcpp_last_total_points", "fcpp_set_profiling", "fcpp_kernel_times", "fcpp_set_cover_mode",
]

_lib = None
_lock = threading.RLock()   # re-entrant: handle() creates a Handle, whose constructor calls load()
_handles = {}


def load():
    """Load libfcpp.so (once).  Raises FcppError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise FcppError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C field_coverage_path_planning_b200/csrc`). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
        L.fcpp_abi_version.restype = C.c_int
        L.fcpp_create.restype = C.c_int
        L.fcpp_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.fcpp_destroy.restype = None
        L.fcpp_destroy.argtypes = [vp]
        L.fcpp_last_error.restype = C.c_char_p
        L.fcpp_last_error.argtypes = [vp]
        L.fcpp_launch_count.restype = i64
        L.fcpp_launch_count.argtypes = [vp]
        L.fcpp_set_trig_tables.restype = C.c_int
        L.fcpp_set_trig_tables.argtypes = [vp, vp, vp, vp, vp]
        L.fcpp_layout.restype = C.c_int
        L.fcpp_layout.argtypes = [vp, C.POINTER(Batch), vp, vp, vp]
        L.fcpp_plan_batch.restype = C.c_int
        L.fcpp_plan_batch.argtypes = [vp, C.POINTER(Batch), C.POINTER(Outputs), vp]
        L.fcpp_obstacle_sweep.restype = C.c_int
        L.fcpp_obstacle_sweep.argtypes = [vp, C.POINTER(Batch), vp, vp]
        L.fcpp_obstacle_sweep_paths.restype = C.c_int
        L.fcpp_obstacle_sweep_paths.argtypes = [vp, vp, vp, i64, vp, vp, vp, i32, dbl, vp, vp]
        L.fcpp_field_select.restype = C.c_int
        L.fcpp_field_select.argtypes = [vp, vp, vp, i64, i32, C.POINTER(SelectionC), i64, vp, vp, vp]
        L.fcpp_field_select_merge.restype = C.c_int
        L.fcpp_field_select_merge.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp]
        L.fcpp_winner_records.restype = C.c_int
        L.fcpp_winner_records.argtypes = [vp, vp, i64, i64, vp, i32, vp, vp]
        L.fcpp_status_count.restype = C.c_int
        L.fcpp_status_count.argtypes = [vp, vp, i64, i32, vp, vp]
        L.fcpp_speed_verify.restype = C.c_int
        L.fcpp_speed_verify.argtypes = [vp, C.POINTER(Vehicle), vp, vp, vp, i64, i64, C.c_int, vp, vp, vp, vp]
        L.fcpp_raster_window.restype = C.c_int
        L.fcpp_raster_window.argtypes = [vp, vp, i32, dbl, dbl, dbl, dbl, i32, vp, vp, vp]
        L.fcpp_tour_lengths.restype = C.c_int
        L.fcpp_tour_lengths.argtypes = [vp, vp, i32, vp, i64, vp, vp, vp]
        L.fcpp_distance_matrix.restype = C.c_int
        L.fcpp_distance_matrix.argtypes = [vp, vp, i32, vp, vp]
        L.fcpp_connection_matrix.restype = C.c_int
        L.fcpp_connection_matrix.argtypes = [vp, vp, i32, dbl, dbl, vp, vp, vp]
        L.fcpp_ga_init_population.restype = C.c_int
        L.fcpp_ga_init_population.argtypes = [vp, C.POINTER(GAConfigC), i32, vp, vp]
        L.fcpp_ga_next_size.restype = i32
        L.fcpp_ga_next_size.argtypes = [C.POINTER(GAConfigC), i32]
        L.fcpp_ga_generation.restype = C.c_int
        L.fcpp_ga_generation.argtypes = [vp, C.POINTER(GAConfigC), i32, i32, vp, vp, i32, vp, vp, vp]
        L.fcpp_ga_solve.restype = C.c_int
        L.fcpp_ga_solve.argtypes = [vp, C.POINTER(GAConfigC), vp, i32, vp, vp, vp, C.POINTER(GAResultC), vp]
        L.fcpp_kmeans_lloyd.restype = C.c_int
        L.fcpp_kmeans_lloyd.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp, i32, dbl, vp, vp, vp]
        L.fcpp_tsp_two_opt.restype = C.c_int
        L.fcpp_tsp_two_opt.argtypes = [vp, i32, vp, vp, vp, i32, vp, vp, vp, i32, vp]
        L.fcpp_last_max_points.restype = i32
        L.fcpp_last_max_points.argtypes = [vp]
        L.fcpp_last_max_head_points.restype = i32
        L.fcpp_last_max_head_points.argtypes = [vp]
        L.fcpp_set_profiling.restype = C.c_int
        L.fcpp_set_profiling.argtypes = [vp, C.c_int]
        L.fcpp_last_total_points.restype = C.c_int64
        L.fcpp_last_total_points.argtypes = [vp]
        L.fcpp_set_cover_mode.restype = C.c_int
        L.fcpp_set_cover_mode.argtypes = [vp, C.c_int]
        L.fcpp_kernel_times.restype = C.c_int
        L.fcpp_kernel_times.argtypes = [vp, C.POINTER(C.c_float * 3)]
        if L.fcpp_abi_version() != ABI_VERSION:
            raise FcppError(f"libfcpp.so ABI {L.fcpp_abi_version()} != expected {ABI_VERSION}: rebuild")
        _lib = L
    return _lib


def trig_tables():
    """cos/sin of the reference's sample angles computed with the SAME numpy calls as the
    reference (mlp3:807-808, :1046-1047), handed to the device so arcs are bit-identical."""
    a20 = np.linspace(0, np.pi, 20)
    a15 = np.linspace(0, np.pi / 2, 15)
    return (np.ascontiguousarray(np.cos(a20)), np.ascontiguousarray(np.sin(a20)),
            np.ascontiguousarray(np.cos(a15)), np.ascontiguousarray(np.sin(a15)))


class Handle:
    """One fcpp_handle per CUDA device (work is enqueued on torch's current stream)."""

    def __init__(self, device_index: int):
        L = load()
        h = C.c_void_p()
        rc = L.fcpp_create(int(device_index), C.byref(h))
        if rc != 0:
            raise FcppError(
                f"fcpp_create(device={device_index}) failed with status {rc}: a CUDA device is required "
                "(this library has no CPU path)")
        self.lib = L
        self.h = h
        self.device_index = int(device_index)
        t = trig_tables()
        self._tables = t
        self.check(L.fcpp_set_trig_tables(h, *[x.ctypes.data for x in t]))

    def check(self, rc: int):
        if rc != 0:
            msg = self.lib.fcpp_last_error(self.h)
            raise FcppError(f"libfcpp status {rc}: {msg.decode() if msg else ''}")

    @property
    def launches(self) -> int:
        return int(self.lib.fcpp_launch_count(self.h))

    def __del__(self):
        try:
            if self.h:
                self.lib.fcpp_destroy(self.h)
                self.h = None
        except Exception:
            pass


def handle(device_index: int = 0, slot: int = 0) -> Handle:
    """The fcpp_handle of a device.  ``slot`` > 0 gives further independent handles (own workspace) for
    work that overlaps slot 0 on another stream (each handle owns its workspace and is not re-entrant)."""
    key = device_index if slot == 0 else (device_index, slot)
    with _lock:
        h = _handles.get(key)
        if h is None:
            h = Handle(device_index)
            _handles[key] = h
    return h
