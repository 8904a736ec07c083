"""efficient_slowfast_b200 -- B200-native (sm_100a) batched clip forward path of weidafeng/Efficient-SlowFast.

Public surface mirrors SlowFast/slowfast/models/__init__.py of the reference:
    from efficient_slowfast_b200 import MODEL_REGISTRY, build_model, get_cfg
"""
from .build import MODEL_REGISTRY, build_model  # noqa: F401
from .config import (CfgNode, ava_slow_8x8_r50_cfg, ava_slowfast_32x2_r50_cfg, get_cfg, resnet_cfg, slowfast_4x16_r50_cfg, slowfast_dual_8x8_r50_cfg,  # noqa: F401
                     slowfast_ghostnet_cfg, slowfast_mobilenetv2_cfg, slowfast_shufflenet_cfg,
                     slowfast_shufflenetv2_cfg)
from .pipeline import ClipStream  # noqa: F401
from .demo import CameraWindows, SlidingWindow  # noqa: F401
from .jpeg import decode_jpeg  # noqa: F401
from .testing import TestMeter, perform_test, topks_correct  # noqa: F401
from .checkpoint import load_checkpoint, save_checkpoint  # noqa: F401
from . import nets_resnet  # noqa: F401  (registers SlowFast, SlowFastDualAttention)
from . import nets_efficient  # noqa: F401  (registers SlowFastShuffleNetV2, SlowFastShuffleNet, ...)

__all__ = ["MODEL_REGISTRY", "build_model", "get_cfg", "CfgNode", "ClipStream", "decode_jpeg", "slowfast_4x16_r50_cfg",
           "slowfast_dual_8x8_r50_cfg"]
