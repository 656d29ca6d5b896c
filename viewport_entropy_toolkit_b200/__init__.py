"""viewport_entropy_toolkit_b200 -- B200-native SpatialEntropyAnalyzer /
TransitionEntropyAnalyzer hot path of viewport-entropy-toolkit.

Same public names as the reference package for the accelerated path; compute runs
in hand-written sm_100a CUDA kernels behind a C ABI (include/vet_b200.h).  Importing
the package does not need a GPU; computing anything does.
"""
from .data_types import Point, RadialPoint, Vector, ValidationError, SpatialError, convert_vectors_to_coordinates
from .config import (AnalyzerConfig, NaiveAnalyzerConfig, EntropyConfig, VisualizationConfig, DEFAULT_VIDEO_DIMENSIONS,
                     DEFAULT_TILE_COUNTS, DEFAULT_OUTPUT_FORMATS)
from .engine import (Engine, SpatialResult, TransitionResult, UserResult, TransitionCountsResult, UserTransitionResult,
                     UnsupportedConfigurationError, get_engine)
from .analyzers import SpatialEntropyAnalyzer, TransitionEntropyAnalyzer, NaiveSpatialEntropyAnalyzer
from .distributed import users_sharded, transition_counts_sharded, user_transitions_sharded
from . import utilities
from .utilities import (generate_fibonacci_lattice, normalize_to_pixel, pixel_to_spherical, validate_video_dimensions,
                        vector_angle_distance, find_angular_distances, find_nearest_tile, calculate_tile_weights,
                        compute_spatial_entropy, compute_transition_entropy,
                        find_naive_tile_index, calculate_naive_tile_weights, compute_naive_spatial_entropy,
                        process_viewport_data, format_trajectory_data)

__version__ = "0.1.0"
__all__ = [
    "Point", "RadialPoint", "Vector", "ValidationError", "SpatialError", "convert_vectors_to_coordinates",
    "AnalyzerConfig", "NaiveAnalyzerConfig", "EntropyConfig", "VisualizationConfig",
    "DEFAULT_VIDEO_DIMENSIONS", "DEFAULT_TILE_COUNTS", "DEFAULT_OUTPUT_FORMATS",
    "Engine", "SpatialResult", "TransitionResult", "UserResult", "TransitionCountsResult", "UserTransitionResult",
    "UnsupportedConfigurationError", "get_engine", "users_sharded", "transition_counts_sharded", "user_transitions_sharded",
    "SpatialEntropyAnalyzer", "TransitionEntropyAnalyzer", "NaiveSpatialEntropyAnalyzer",
    "generate_fibonacci_lattice", "normalize_to_pixel", "pixel_to_spherical", "validate_video_dimensions",
    "vector_angle_distance", "find_angular_distances", "find_nearest_tile", "calculate_tile_weights",
    "compute_spatial_entropy", "compute_transition_entropy",
    "find_naive_tile_index", "calculate_naive_tile_weights", "compute_naive_spatial_entropy",
    "process_viewport_data", "format_trajectory_data",
]
