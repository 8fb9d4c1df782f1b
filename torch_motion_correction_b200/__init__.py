"""B200-native drop-in for the hot path of ``torch_motion_correction``.

Same public names, argument meaning, tensor shapes and spline-grid outputs as the reference
package (``/root/reference/src/torch_motion_correction/__init__.py:12-44``); every kernel is
hand-written CUDA for sm_100a behind a C ABI (``include/tmc_b200.h``).  No CPU fallback.
"""

from .correct_motion import (
    correct_motion,
    correct_motion_fast,
    correct_motion_slow,
    correct_motion_sum,
    correct_motion_sums,
    correct_motion_two_grids,
    get_pixel_shifts,
)
from .deformation_field_utils import (
    evaluate_deformation_field,
    evaluate_deformation_field_at_t,
    image_shifts_to_deformation_field,
    resample_deformation_field,
)

from .dose_weight import dose_weight
from .data_io import read_deformation_field_from_csv, write_deformation_field_to_csv
from .estimate_motion_optimizer import estimate_local_motion
from .estimate_motion_xc import estimate_global_motion, estimate_motion_cross_correlation_patches
from .optimization_state import OptimizationState, OptimizationTracker
from .patch_grid import patch_grid_centers
from .spline_grids import CubicBSplineGrid3d, CubicCatmullRomGrid3d
from .pipeline import estimate_motion, motion_correct, motion_correct_many
from .prepare import fourier_crop, group_frames, prepare_movie, render_eer
from .movie_io import EerMovie, eer_movies, mrc_movies, read_eer, read_mrc, read_mrc_header, read_tiff, write_mrc
from .utils import normalize_image

__version__ = "0.1.0"

__all__ = [
    "estimate_local_motion",
    "write_deformation_field_to_csv",
    "read_deformation_field_from_csv",
    "correct_motion",
    "correct_motion_two_grids",
    "correct_motion_fast",
    "correct_motion_slow",
    "correct_motion_sum",
    "correct_motion_sums",
    "get_pixel_shifts",
    "evaluate_deformation_field",
    "estimate_global_motion",
    "estimate_motion_cross_correlation_patches",
    "estimate_motion",
    "motion_correct",
    "motion_correct_many",
    "dose_weight",
    "prepare_movie",
    "group_frames",
    "fourier_crop",
    "read_mrc",
    "read_mrc_header",
    "write_mrc",
    "mrc_movies",
    "render_eer",
    "read_eer",
    "eer_movies",
    "read_tiff",
    "EerMovie",
]
