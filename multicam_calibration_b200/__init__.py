"""B200-native bundle-adjustment engine behind the Python API of
``multicam_calibration.bundle_adjustment`` and ``multicam_calibration.geometry``.

``import multicam_calibration_b200 as mcc`` exposes the same flat namespace the
reference builds with its star imports (``multicam_calibration/__init__.py:1-7``)
for the two hot-path modules, plus the steps on either side of them: the rigid-transform part of
``calibration`` that produces bundle_adjust's initial guess (calibration.py:116-277), the
reprojection-error check of its result (viz.py:70-210) and the calibration files (io.py:8-245), the
covariance of a calibration (``calibration_covariance``: what a reference user derives from ``result.jac``), and
the least-squares refinement of triangulated points (``refine_points``).
"""
from .geometry import (rodrigues, rodrigues_inv, rigid_transform_from_correspondences,
                       apply_rigid_transform, get_transformation_matrix, get_transformation_vector,
                       get_projection_matrix, euclidean_to_homogenous, homogeneous_to_euclidean,
                       project_points, project_points_multi, undistort_points, triangulate,
                       refine_points, RefinedPoints)
from .bundle_adjustment import (embed_calib_objpoints, predict_calib_uvs, residuals,
                                bundle_adjustment_sparsity, serialize_params, deserialize_params,
                                bundle_adjust, select_frames)
from .bundle_adjustment import release_device_memory
from .calibration import (estimate_pairwise_camera_transform, get_camera_spanning_tree,
                          estimate_all_extrinsics, consensus_calib_poses)
from .io import save_calibration, load_calibration
from .viz import plot_residuals, reprojection_residuals
from .engine import BAProblem, OptimizeResult
from .covariance import calibration_covariance, CalibrationCovariance, point_covariance, PointCovariance

__version__ = "0.1.0"
