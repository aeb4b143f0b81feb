"""ekf-slam-ml_b200 — B200-native EKF-SLAM hot path (rigid2d::EKF_SLAM + rigid2d::CircleFitting).

The directory name carries a hyphen (it mirrors the reference repo's name), so import it through the
root-level shim:  ``import ekf_slam_ml_b200``.
"""
from . import _lib, consistency, report, sharding, tracegen
from ._lib import EkfError, device_count
from .circle_fitting import CircleFitting
from .tube_world import TubeWorld
from .ekf_slam import (DiffDrive, EKF_SLAM, ENGINE_AUTO, ENGINE_FUSED, ENGINE_STREAM, EKFBatch, PinnedBuffer, Twist2D,
                       Vector2D, body_twist, marker_list, normalize_angle, update_pose)

__all__ = ["DiffDrive", "update_pose", "EKF_SLAM", "EKFBatch", "PinnedBuffer", "Twist2D", "Vector2D", "body_twist", "marker_list", "normalize_angle",
           "EkfError", "device_count", "tracegen", "sharding", "report", "consistency", "CircleFitting", "TubeWorld", "ENGINE_AUTO", "ENGINE_FUSED", "ENGINE_STREAM"]
