"""aruco3_b200 — B200-native (sm_100a) detection front end and tag decode of aruco3.

The product is `libaruco3_b200.so` (C ABI in include/aruco3_b200.h); this package is its host-side mirror of
the reference interface (`Detector { config, dictionary }.detect(img)`), the marker tables and the synthetic
workload generator.  No CPU fallback exists anywhere in this package.
"""
from .detector import (ARDictionary, Detection, Detector, DetectorConfig, Marker, hamming_distance,  # noqa: F401
                       quads_from_mask)
from ._ffi import A3Error  # noqa: F401
from . import pose  # noqa: F401
from .pose import CameraDistortion, CameraIntrinsics, MarkerPose  # noqa: F401
from .board import Board, BoardPose  # noqa: F401

__version__ = "0.1.0"
