"""B200-native batched plan generation + validation for the two-layer field coverage planner.

Drop-in for the hot path of qwagrox/field-coverage-path-planning (SURVEY.md §8): the reference's
class API on top of hand-written sm_100a CUDA kernels behind a C-ABI (include/fcpp.h).
No CPU fallback: importing works anywhere, computing needs libfcpp.so and a CUDA device.
"""
from .vehicle import VehicleParams  # noqa: F401
from ._lib import FcppError  # noqa: F401
from .batch import (BatchResult, Selection, candidate_axes, expand_axes, make_candidates, obstacle_sweep,  # noqa: F401
                    plan_batch, prepare_batch, verify_paths)
from .planner import (TwoLayerPathPlannerV35, TwoLayerPathPlannerV36, TwoLayerPathPlannerV37,  # noqa: F401
                      TwoLayerPlannerV35, TwoLayerPlannerV36, TwoLayerPlannerV37)
from .ga import GAConfig, GeneticAlgorithmSolver, tour_lengths  # noqa: F401
from .multi_field import (Connection, FieldData, MultiFieldPlannerV38, OptimizedRoute,  # noqa: F401
                          connection_matrix, distance_matrix)

from .multi_vehicle import MultiVehiclePlanner, MultiVehicleRoute, VehicleRoute, kmeans_labels  # noqa: F401

from .tsp import TSPSolver, two_opt_batch  # noqa: F401

__all__ = ["TSPSolver", "two_opt_batch", "MultiVehiclePlanner", "MultiVehicleRoute", "VehicleRoute", "kmeans_labels", "VehicleParams", "TwoLayerPathPlannerV37", "TwoLayerPathPlannerV35", "TwoLayerPathPlannerV36",
           "TwoLayerPlannerV35", "TwoLayerPlannerV36", "TwoLayerPlannerV37", "plan_batch", "prepare_batch",
           "make_candidates", "candidate_axes", "obstacle_sweep", "verify_paths", "Selection", "expand_axes", "BatchResult", "tour_lengths", "GeneticAlgorithmSolver", "GAConfig", "FcppError",
           "MultiFieldPlannerV38", "FieldData", "Connection", "OptimizedRoute", "distance_matrix",
           "connection_matrix"]
