"""feature_extraction_b200 — B200-native per-scan keypoint pipeline (drop-in for the processing
callback of GAVLab/feature_extraction, reference src/feature_extraction_node.cpp:83-117).

The compute path is csrc/libfe_b200.so (hand-written sm_100a CUDA behind the C-ABI of
include/fe_b200.h); this package is only the host-side mirror of the reference's interface.
"""
from .node import (FeatureExtractionNode, MultiGpuExtractor, FeatureExtractionError, PinnedBuffer, node_default,  # noqa: F401
                   launch_playback, register_params_default, loop_params_default, rotation_matrix, imu_to_roll_pitch, pack_point_descriptors, DESC_LEN,
                   ODOMETRY_WINDOW)
