"""dynamic_vins_b200 — B200-native feature-tracking front-end (Dynamic-VINS hot path).

The compute path is libdvfe.so (hand-written sm_100a CUDA kernels behind the C ABI of include/dvfe.h).
This package is the thin host-side mirror of the reference's FeatureTracker interface over that ABI.
"""
from . import synth  # noqa: F401  (numpy only)
from ._lib import DvfeError, LIB_PATH, lib, FRAME_SKIP, FRAME_NO_RIGHT, FRAME_RESET, STEP_DEVICE_INPUT  # noqa: F401
from .tracker import BatchTracker, FeatureTracker, Frame, camera_from_yaml, config_from_yaml, make_config, obs_to_map  # noqa: F401
from . import ops  # noqa: F401

__all__ = ["BatchTracker", "FeatureTracker", "Frame", "camera_from_yaml", "config_from_yaml", "make_config", "obs_to_map", "ops", "synth",
           "DvfeError", "lib", "LIB_PATH", "FRAME_SKIP", "FRAME_NO_RIGHT", "FRAME_RESET", "STEP_DEVICE_INPUT"]
