"""Config tree for the clip forward path.

Same key names and defaults as the reference's yacs tree for every key the model builders read
(SlowFast/slowfast/config/defaults.py:100-260,343,403,502 and custom_config.py:11-35; the list of keys on this
path is SURVEY.md section 8b).  Any attribute-style cfg object with these keys is accepted by build_model(),
including the reference's own CfgNode -- this class only exists so the package has no yacs/fvcore dependency.
"""
import ast
import copy

import yaml


class CfgNode(dict):
    def __init__(self, d=None):
        super().__init__()
        for k, v in (d or {}).items():
            self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __setattr__(self, k, v):
        self[k] = v

    def clone(self):
        return copy.deepcopy(self)

    def _merge(self, other):
        for k, v in other.items():
            if isinstance(v, dict) and isinstance(self.get(k), dict):
                self[k]._merge(v)
            else:
                self[k] = CfgNode(v) if isinstance(v, dict) else v

    def merge_from_file(self, path):
        with open(path) as fh:
            self._merge(yaml.safe_load(fh) or {})

    def merge_from_list(self, lst):
        assert len(lst) % 2 == 0, "merge_from_list expects KEY VALUE pairs"
        for k, v in zip(lst[0::2], lst[1::2]):
            node, ks = self, k.split(".")
            for kk in ks[:-1]:
                node = node[kk]
            if isinstance(v, str):
                try:
                    v = ast.literal_eval(v)
                except (ValueError, SyntaxError):
                    pass
            node[ks[-1]] = v


def get_cfg():
    """Defaults of the keys on the forward path (reference: config/defaults.py:639-643 get_cfg)."""
    c = CfgNode()
    c.BN = CfgNode(dict(NORM_TYPE="batchnorm", NUM_SPLITS=1, NUM_SYNC_DEVICES=1))
    c.RESNET = CfgNode(dict(
        TRANS_FUNC="bottleneck_transform", NUM_GROUPS=1, WIDTH_PER_GROUP=64, INPLACE_RELU=True, STRIDE_1X1=False,
        ZERO_INIT_FINAL_BN=False, DEPTH=50, NUM_BLOCK_TEMP_KERNEL=[[3], [4], [6], [3]],
        SPATIAL_STRIDES=[[1], [2], [2], [2]], SPATIAL_DILATIONS=[[1], [1], [1], [1]]))
    c.NONLOCAL = CfgNode(dict(
        LOCATION=[[[]], [[]], [[]], [[]]], GROUP=[[1], [1], [1], [1]], INSTANTIATION="dot_product",
        POOL=[[[1, 2, 2], [1, 2, 2]]] * 4))
    c.MODEL = CfgNode(dict(ARCH="slowfast", MODEL_NAME="SlowFast", NUM_CLASSES=400, LOSS_FUNC="cross_entropy",
                           DROPOUT_RATE=0.5, FC_INIT_STD=0.01, HEAD_ACT="softmax"))
    c.SLOWFAST = CfgNode(dict(BETA_INV=8, ALPHA=8, FUSION_CONV_CHANNEL_RATIO=2, FUSION_KERNEL_SZ=5,
                              WIDTH_MULTI=2.0, GROUPS=1))
    c.DATA = CfgNode(dict(NUM_FRAMES=8, CROP_SIZE=224, TRAIN_CROP_SIZE=224, TEST_CROP_SIZE=256,
                          INPUT_CHANNEL_NUM=[3, 3], MEAN=[0.45, 0.45, 0.45], STD=[0.225, 0.225, 0.225],
                          SAMPLING_RATE=8, TARGET_FPS=30, REVERSE_INPUT_CHANNEL=False))
    c.DETECTION = CfgNode(dict(ENABLE=False, ALIGNED=True, ROI_XFORM_RESOLUTION=7, SPATIAL_SCALE_FACTOR=16))
    c.MULTIGRID = CfgNode(dict(SHORT_CYCLE=False, LONG_CYCLE=False))
    c.TEST = CfgNode(dict(BATCH_SIZE=8, NUM_ENSEMBLE_VIEWS=10, NUM_SPATIAL_CROPS=3))
    c.NUM_GPUS = 1
    # extension (not in the reference): 16-bit storage / tensor-core operand format of the CUDA path, "bf16" or "fp16"
    # (FP32 accumulation, softmax statistics and head in both; fp16 has 3 more mantissa bits and saturates at 65504)
    c.ESF = CfgNode(dict(PRECISION="fp16", CUDA_GRAPH=True))
    return c


# The two ResNet-50 YAMLs named by BASELINE.json, restated as overrides of get_cfg()
# (SlowFast/configs/Kinetics/SLOWFAST_4x16_R50.yaml, SLOWFAST_DUAL_8x8_R50_stepwise_multigrid.yaml).
_R50_TWO_PATH = dict(
    ZERO_INIT_FINAL_BN=True, WIDTH_PER_GROUP=64, NUM_GROUPS=1, DEPTH=50, TRANS_FUNC="bottleneck_transform",
    STRIDE_1X1=False, NUM_BLOCK_TEMP_KERNEL=[[3, 3], [4, 4], [6, 6], [3, 3]],
    SPATIAL_STRIDES=[[1, 1], [2, 2], [2, 2], [2, 2]], SPATIAL_DILATIONS=[[1, 1], [1, 1], [1, 1], [1, 1]])
_NONLOCAL_OFF = dict(LOCATION=[[[], []], [[], []], [[], []], [[], []]], GROUP=[[1, 1], [1, 1], [1, 1], [1, 1]],
                     INSTANTIATION="dot_product")


def slowfast_4x16_r50_cfg():
    c = get_cfg()
    c.RESNET._merge(_R50_TWO_PATH)
    c.NONLOCAL._merge(_NONLOCAL_OFF)
    c.DATA._merge(dict(NUM_FRAMES=32, INPUT_CHANNEL_NUM=[3, 3]))
    c.SLOWFAST._merge(dict(ALPHA=8, BETA_INV=8, FUSION_CONV_CHANNEL_RATIO=2, FUSION_KERNEL_SZ=5))
    c.MODEL._merge(dict(NUM_CLASSES=400, ARCH="slowfast", MODEL_NAME="SlowFast", DROPOUT_RATE=0.5))
    return c


def slowfast_dual_8x8_r50_cfg():
    c = get_cfg()
    c.RESNET._merge(_R50_TWO_PATH)
    c.NONLOCAL._merge(_NONLOCAL_OFF)
    c.DATA._merge(dict(NUM_FRAMES=32, INPUT_CHANNEL_NUM=[3, 3]))
    c.SLOWFAST._merge(dict(ALPHA=4, BETA_INV=8, FUSION_CONV_CHANNEL_RATIO=2, FUSION_KERNEL_SZ=7, WIDTH_MULTI=0.25))
    c.MODEL._merge(dict(NUM_CLASSES=400, ARCH="slowfast", MODEL_NAME="SlowFastDualAttention", DROPOUT_RATE=0.5))
    c.MULTIGRID._merge(dict(SHORT_CYCLE=True, LONG_CYCLE=True))
    return c


def resnet_cfg(arch="i3d", num_frames=8, nln=False):
    """configs/Kinetics/{C2D,I3D,SLOW}_8x8_R50.yaml: single-pathway ResNet-50, MODEL_NAME ResNet, ARCH c2d / i3d / slow."""
    c = get_cfg()
    c.RESNET._merge(dict(ZERO_INIT_FINAL_BN=True, WIDTH_PER_GROUP=64, NUM_GROUPS=1, DEPTH=50,
                         TRANS_FUNC="bottleneck_transform", STRIDE_1X1=False,
                         NUM_BLOCK_TEMP_KERNEL=[[3], [4], [6], [3]], SPATIAL_STRIDES=[[1], [2], [2], [2]],
                         SPATIAL_DILATIONS=[[1], [1], [1], [1]]))
    # nln: configs/Kinetics/{C2D,I3D,SLOW}_NLN_8x8_R50.yaml
    c.NONLOCAL._merge(dict(LOCATION=[[[]], [[1, 3]], [[1, 3, 5]], [[]]] if nln else [[[]], [[]], [[]], [[]]],
                           GROUP=[[1], [1], [1], [1]],
                           INSTANTIATION="softmax" if arch != "slow" else "dot_product"))
    c.DATA._merge(dict(NUM_FRAMES=num_frames, INPUT_CHANNEL_NUM=[3]))
    c.MODEL._merge(dict(NUM_CLASSES=400, ARCH=arch, MODEL_NAME="ResNet", DROPOUT_RATE=0.5))
    return c


def _ava_cfg(c):
    """What the AVA detection YAMLs of upstream SlowFast (configs/AVA/SLOWFAST_32x2_R50_SHORT.yaml,
    SLOW_8x8_R50_SHORT.yaml) set on top of the Kinetics R50 models: the RoI head, 80 sigmoid classes and res5 at spatial
    stride 1 with dilation 2 (feature stride 16, DETECTION.SPATIAL_SCALE_FACTOR).  The values are restated from the
    upstream files; the fork's copies of these YAMLs could not be read when this was written, and
    tests/test_detection.py::test_ava_yamls_match_reference compares them wherever the reference tree is available."""
    npw = len(c.DATA.INPUT_CHANNEL_NUM)
    c.RESNET._merge(dict(SPATIAL_STRIDES=[[1] * npw, [2] * npw, [2] * npw, [1] * npw],
                         SPATIAL_DILATIONS=[[1] * npw, [1] * npw, [1] * npw, [2] * npw]))
    c.DETECTION._merge(dict(ENABLE=True, ALIGNED=True, ROI_XFORM_RESOLUTION=7, SPATIAL_SCALE_FACTOR=16))
    c.MODEL._merge(dict(NUM_CLASSES=80, HEAD_ACT="sigmoid"))
    c.DATA._merge(dict(TRAIN_CROP_SIZE=224, TEST_CROP_SIZE=256))
    return c


def ava_slowfast_32x2_r50_cfg():
    """configs/AVA/SLOWFAST_32x2_R50_SHORT.yaml: SlowFast R50, 32 fast / 8 slow frames (ALPHA 4), fusion kernel 7."""
    c = slowfast_4x16_r50_cfg()
    c.DATA._merge(dict(NUM_FRAMES=32, SAMPLING_RATE=2))
    c.SLOWFAST._merge(dict(ALPHA=4, BETA_INV=8, FUSION_CONV_CHANNEL_RATIO=2, FUSION_KERNEL_SZ=7))
    return _ava_cfg(c)


def ava_slow_8x8_r50_cfg():
    """configs/AVA/SLOW_8x8_R50_SHORT.yaml: single-pathway Slow R50, 8 frames."""
    c = resnet_cfg("slow", num_frames=8)
    return _ava_cfg(c)


def _efficient_cfg(model_name, width_multi, groups=1, num_classes=400, num_frames=16, crop=112, dropout=0.5,
                   short_cycle=True):
    """Shared part of the four efficient YAMLs (configs/Kinetics/SLOWFAST_{SHUFFLENETV2,MOBILENETV2,GHOSTNET}_8x8_*.yaml,
    configs/Jester/SLOWFAST_SHUFFLENET_8x8_*.yaml): NUM_FRAMES 16, ALPHA 4, BETA_INV 8, crop 112."""
    c = get_cfg()
    c.RESNET._merge(_R50_TWO_PATH)
    c.NONLOCAL._merge(_NONLOCAL_OFF)
    c.DATA._merge(dict(NUM_FRAMES=num_frames, INPUT_CHANNEL_NUM=[3, 3], CROP_SIZE=crop, TRAIN_CROP_SIZE=crop,
                       TEST_CROP_SIZE=crop))
    c.SLOWFAST._merge(dict(ALPHA=4, BETA_INV=8, FUSION_CONV_CHANNEL_RATIO=2, FUSION_KERNEL_SZ=7,
                           WIDTH_MULTI=width_multi, GROUPS=groups))
    c.MODEL._merge(dict(NUM_CLASSES=num_classes, ARCH="slowfast", MODEL_NAME=model_name, DROPOUT_RATE=dropout))
    c.MULTIGRID._merge(dict(SHORT_CYCLE=short_cycle, LONG_CYCLE=short_cycle))
    return c


def slowfast_shufflenetv2_cfg(width_multi=2.0):
    return _efficient_cfg("SlowFastShuffleNetV2", width_multi, short_cycle=False)


def slowfast_shufflenet_cfg(width_multi=2.0, groups=3):
    """Jester YAML: 27 classes, dropout 0.2."""
    return _efficient_cfg("SlowFastShuffleNet", width_multi, groups=groups, num_classes=27, dropout=0.2)


def slowfast_mobilenetv2_cfg(width_multi=0.5):
    return _efficient_cfg("SlowFastMoibleNetV2", width_multi)


def slowfast_ghostnet_cfg(width_multi=1.0):
    return _efficient_cfg("SlowFastGhostNet", width_multi)
