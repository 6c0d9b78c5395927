"""icet_b200 -- B200-native (sm_100a) implementation of ICET's per-scan-pair registration hot path.

Python host-side mirror of the reference interface (`class ICET`, reference include/icet.h:36-116)
over the C ABI of include/icet_b200.h.  There is no CPU fallback: importing works anywhere, but
every compute entry point raises if the CUDA library or a B200 is missing.
"""
from .api import ICET, Context, IcetError, Keyframe, MultiContext, Params, Result, lib_path, load_library  # noqa: F401
from .build import build  # noqa: F401
from .nodes import KeyframeOdometryNode, MapMakerNode, Node, OdometryNode, PointMap, ScanMatcherNode  # noqa: F401

__all__ = ["ICET", "Context", "Keyframe", "MultiContext", "IcetError", "Params", "Result", "build", "load_library", "lib_path",
           "OdometryNode", "MapMakerNode", "ScanMatcherNode", "Node", "PointMap", "KeyframeOdometryNode"]
