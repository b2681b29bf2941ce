"""tepose_b200 -- B200-native (sm_100a) implementation of TePose's per-sequence inference hot
path behind the reference's lib.models API.  See DESIGN.md / INTEGRATION.md."""
from .tepose import TePose, TemporalEncoder  # noqa: F401
from .vibe import VIBE  # noqa: F401
from .spin import Regressor, projection  # noqa: F401
from .hmr import HMR, hmr  # noqa: F401
from .video import VideoTePose  # noqa: F401
from .tracks import TrackedTePose, TrackedVideoTePose  # noqa: F401
from .render import MeshRenderer, crop_cam_to_frame, crop_kp_to_frame, render_clip  # noqa: F401
from .smooth import smooth_pose  # noqa: F401
from .smpl import (SMPL, SMPLOutput, JOINT_MAP, JOINT_NAMES, JOINT_IDS, H36M_TO_J14, H36M_TO_J17,  # noqa: F401
                   SMPL_MODEL_DIR, SMPL_MEAN_PARAMS, BASE_DATA_DIR, get_smpl_faces)
from .geometry import rot6d_to_rotmat, rotation_matrix_to_angle_axis, batch_rodrigues  # noqa: F401

__version__ = "0.1.0"
