"""amodal-depth-anything_b200: B200 (sm_100a) implementation of the discriminative forward pass of
Amodal-Depth-Anything behind the reference's own Python model API.

The directory name carries a hyphen (it mirrors the reference repo name); import it as `amodal_depth_anything_b200`
(the shim of that name at the repo root loads this package).
"""
from . import _lib  # noqa: F401  (ctypes binding; loading the .so is deferred to first use)
from .evaluate import AmodalEvaluator  # noqa: F401
from .infer import AmodalInference  # noqa: F401
from .model import GUIDE_CHANNELS, MODEL_CONFIGS, AmodalDAv2, DepthAnythingV2, get_model  # noqa: F401

__all__ = ["AmodalDAv2", "DepthAnythingV2", "AmodalInference", "AmodalEvaluator", "get_model", "MODEL_CONFIGS", "GUIDE_CHANNELS", "_lib"]
