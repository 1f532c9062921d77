"""B200-native velocity-measurement hot path (pyramid -> Shi-Tomasi -> pyramidal LK -> planar-flow
least squares -> Monte-Carlo error propagation) behind the reference's own Python call shapes.

The directory name follows the repository naming rule and is not a Python identifier; import the
package through the `ofb200` alias module at the repository root:

    import ofb200
    import ofb200.of_library as of          # drop-in for the reference's of_library
    from ofb200 import solve_lgs, goodFeaturesToTrack, calcOpticalFlowPyrLK

Everything computes in libofb200.so (hand-written sm_100a CUDA, C ABI in include/ofb200.h). There is
no CPU fallback: without the built library or without a B200 every call raises.
"""
from . import _lib
from ._lib import Context, OfbError, default_context
from . import of_library, velocity, vision, simulation, tracker, replay
from .of_library import pix_trans, r_tilde, static_immobile, initialize_ft
from .velocity import (solve_lgs, solve_full, solve_lgs_batched, solve_lgs_module, generate_test_data, feasibility,
                       quaternion_to_rotation, plane_normal, body_to_world, solve_ego_motion, solve_ego_motion_batched,
                       solve_velocity_robust, solve_velocity_robust_batched)
from .vision import (goodFeaturesToTrack, calcOpticalFlowPyrLK, cornerMinEigenVal, buildPyramid, pyrDown, cvtColor,
                     Pyramid, make_pair_cfg, frame_pairs, frame_sequence, COLOR_BGR2GRAY, TERM_CRITERIA_COUNT, TERM_CRITERIA_EPS,
                     undistortPoints, undistortPointsIter, make_camera, CAMERA_ITERATIONS, track_forward_backward,
                     gyro_predict)
from .tracker import StreamTracker, FleetTracker, exclusion_mask
from .simulation import of_simulation, feas_simulation, overlap, run_named_sweep, run_sweep, sorting_study, advect_points

__version__ = "0.1.0"
