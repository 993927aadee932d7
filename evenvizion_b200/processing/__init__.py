"""Drop-in for `evenvizion.processing` (reference evenvizion/processing/__init__.py): same module
and function names, arithmetic on the GPU through libevz.so."""
__all__ = ['constants', 'frame_processing', 'fixed_coordinate_system', 'formats', 'matching', 'utils', 'video_processing']

from .constants import *                      # noqa: F401,F403
from .frame_processing import FrameProcessing, resize           # noqa: F401
from .fixed_coordinate_system import from_original_to_fix, from_fix_to_original   # noqa: F401
from .matching import KeyPoints, NoMatchesException, lowes_ratio_test, filter_corresponding_points   # noqa: F401
from .utils import (HomographyException, remove_double_matching, homography_transformation,      # noqa: F401
                    inverse_homography_transformation, matrix_superposition, read_homography_dict,
                    superposition_dict, are_infinity_coordinates, read_json_with_coordinates,
                    get_largest_group_points, find_point_displacement, compute_homography)
from .video_processing import (get_homography_dict, get_homography_dicts, geometry_from_features,      # noqa: F401
                               geometry_from_features_batch, read_and_describe)
from .formats import dump_homography_dict, load_homography_arrays, dump_coordinates, load_coordinates_arrays   # noqa: F401
