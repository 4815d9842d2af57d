"""b200seg -- B200 (sm_100a) drop-in for the segmentation hot path of SEAME-pt/Team02-ObjectDetection.

    from b200seg import MobileNetV2UNet, UNet          # same ctor / forward / state_dict as src/unet.py

Importing this package loads ``libb200seg.so`` (hand-written CUDA behind a C ABI, include/b200seg.h).
It raises ImportError if the library has not been built -- there is no eager / CPU fallback.
"""
from . import _cabi  # noqa: F401  (fail loudly if the CUDA library is missing)
from .unet import LightUNet, MobileNetV2UNet, UNet  # noqa: F401
from .loss import CrossEntropyLoss  # noqa: F401
from .optim import Adam  # noqa: F401
from .preprocess import preprocess_image  # noqa: F401
from .feed import DeviceFeeder, class_map_lut, remap_labels  # noqa: F401
from .export import torch_graph  # noqa: F401
from .metrics import SegmentationMetrics  # noqa: F401
from .postprocess import Detections, detect_objects, overlay  # noqa: F401

__all__ = ["MobileNetV2UNet", "UNet", "LightUNet", "CrossEntropyLoss", "Adam", "preprocess_image", "DeviceFeeder",
           "class_map_lut", "remap_labels", "torch_graph", "SegmentationMetrics", "detect_objects", "Detections", "overlay"]
__version__ = "0.1.0"
