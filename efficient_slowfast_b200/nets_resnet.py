"""The two ResNet-50 based two-stream models, behind the reference's registry / nn.Module surface:

  SlowFastDualAttention   (reference: SlowFast/slowfast/models/custom_video_model_builder.py:171-445)
  SlowFast                (reference: SlowFast/slowfast/models/video_model_builder.py:153-416)

The module tree only *holds parameters* under the reference's state_dict keys (SURVEY.md Appendix D), child names
and child order, so checkpoints, BN scans and `load_state_dict` written against the reference keep working.  The
arithmetic is not in these modules: `forward([slow, fast])` compiles (once per input shape) a launch plan of
hand-written sm_100a kernels (engine.py, csrc/) and replays it.  Eval mode only -- the training path (batch-stat BN,
autograd) is outside the hot path this package accelerates and raises.
"""
import collections
import itertools
import math

import torch
import torch.nn as nn

from . import runtime as rt
from .build import MODEL_REGISTRY
from .engine import Family, Plan, fold_conv_bn

# video_model_builder.py:16-90 / custom_video_model_builder.py:151-168
_MODEL_STAGE_DEPTH = {50: (3, 4, 6, 3), 101: (3, 4, 23, 3), 18: (2, 2, 2, 2), 34: (3, 4, 6, 3)}   # 18 / 34: the fork's additions
_TEMPORAL_KERNEL_BASIS = {     # video_model_builder.py:20-75
    "c2d": [[[1]], [[1]], [[1]], [[1]], [[1]]],
    "c2d_nopool": [[[1]], [[1]], [[1]], [[1]], [[1]]],
    "i3d": [[[5]], [[3]], [[3, 1]], [[3, 1]], [[1, 3]]],
    "i3d_nopool": [[[5]], [[3]], [[3, 1]], [[3, 1]], [[1, 3]]],
    "slow": [[[1]], [[1]], [[1]], [[3]], [[3]]],
    "slowfast": [[[1], [5]], [[1], [3]], [[1], [3]], [[3], [3]], [[3], [3]]],
    "fast": [[[5]], [[3]], [[3]], [[3]], [[3]]],      # the fork's single-pathway "fast" arch (video_model_builder.py:79-85)
}
_POOL1 = {"c2d": [[2, 1, 1]], "c2d_nopool": [[1, 1, 1]], "i3d": [[2, 1, 1]], "i3d_nopool": [[1, 1, 1]],
          "slow": [[1, 1, 1]], "slowfast": [[1, 1, 1], [1, 1, 1]], "fast": [[1, 1, 1]]}


class _Holder(nn.Module):
    """Parameter container; the computation happens in the model-level launch plan."""

    def forward(self, *a, **k):
        raise RuntimeError("%s only holds parameters; call the model's forward([slow, fast])" % type(self).__name__)


def get_norm(cfg):
    """batchnorm_helper.py:15-34.  Only plain BatchNorm3d exists on the eval forward path; the sub-/sync-BN variants
    differ from it in training mode only and store the same parameters."""
    if cfg.BN.NORM_TYPE in ("batchnorm", "sub_batchnorm", "sync_batchnorm"):
        return nn.BatchNorm3d
    raise NotImplementedError("Norm type {} is not supported".format(cfg.BN.NORM_TYPE))


# --------------------------------------------------------------------------------------------- holders
class ResNetBasicStem(_Holder):
    """stem_helper.py:102-178: conv kxkxk s(1,2,2) -> BN -> ReLU -> MaxPool (1,3,3) s(1,2,2) p(0,1,1)."""

    def __init__(self, dim_in, dim_out, kernel, stride, padding, norm_module, eps=1e-5, bn_mmt=0.1):
        super().__init__()
        self.kernel, self.stride, self.padding = kernel, stride, padding
        self.conv = nn.Conv3d(dim_in, dim_out, kernel, stride=stride, padding=padding, bias=False)
        self.bn = norm_module(num_features=dim_out, eps=eps, momentum=bn_mmt)
        self.relu = nn.ReLU(True)
        self.pool_layer = nn.MaxPool3d(kernel_size=[1, 3, 3], stride=[1, 2, 2], padding=[0, 1, 1])


class VideoModelStem(_Holder):
    """stem_helper.py:9-99."""

    def __init__(self, dim_in, dim_out, kernel, stride, padding, norm_module):
        super().__init__()
        assert len({len(dim_in), len(dim_out), len(kernel), len(stride), len(padding)}) == 1, \
            "Input pathway dimensions are not consistent."
        self.num_pathways = len(dim_in)
        for p in range(self.num_pathways):
            self.add_module("pathway{}_stem".format(p),
                            ResNetBasicStem(dim_in[p], dim_out[p], kernel[p], stride[p], padding[p], norm_module))


class BottleneckTransform(_Holder):
    """resnet_helper.py:110-240: Tx1x1 -> BN -> ReLU -> 1x3x3 (stride) -> BN -> ReLU -> 1x1x1 -> BN."""

    def __init__(self, dim_in, dim_out, temp_kernel_size, stride, dim_inner, num_groups, stride_1x1, dilation,
                 norm_module, eps=1e-5, bn_mmt=0.1):
        super().__init__()
        str1x1, str3x3 = (stride, 1) if stride_1x1 else (1, stride)
        self.a = nn.Conv3d(dim_in, dim_inner, kernel_size=[temp_kernel_size, 1, 1], stride=[1, str1x1, str1x1],
                           padding=[int(temp_kernel_size // 2), 0, 0], bias=False)
        self.a_bn = norm_module(num_features=dim_inner, eps=eps, momentum=bn_mmt)
        self.a_relu = nn.ReLU(inplace=True)
        self.b = nn.Conv3d(dim_inner, dim_inner, [1, 3, 3], stride=[1, str3x3, str3x3],
                           padding=[0, dilation, dilation], groups=num_groups, bias=False,
                           dilation=[1, dilation, dilation])
        self.b_bn = norm_module(num_features=dim_inner, eps=eps, momentum=bn_mmt)
        self.b_relu = nn.ReLU(inplace=True)
        self.c = nn.Conv3d(dim_inner, dim_out, kernel_size=[1, 1, 1], stride=[1, 1, 1], padding=[0, 0, 0], bias=False)
        self.c_bn = norm_module(num_features=dim_out, eps=eps, momentum=bn_mmt)
        self.c_bn.transform_final_bn = True


class ResBlock(_Holder):
    """resnet_helper.py:243-358."""

    def __init__(self, dim_in, dim_out, temp_kernel_size, stride, dim_inner, num_groups, stride_1x1, dilation,
                 norm_module, eps=1e-5, bn_mmt=0.1):
        super().__init__()
        if (dim_in != dim_out) or (stride != 1):
            self.branch1 = nn.Conv3d(dim_in, dim_out, kernel_size=1, stride=[1, stride, stride], padding=0, bias=False,
                                     dilation=1)
            self.branch1_bn = norm_module(num_features=dim_out, eps=eps, momentum=bn_mmt)
        self.branch2 = BottleneckTransform(dim_in, dim_out, temp_kernel_size, stride, dim_inner, num_groups,
                                           stride_1x1, dilation, norm_module)
        self.relu = nn.ReLU(True)


class Nonlocal(_Holder):
    """nonlocal_helper.py:10-103 (parameter holder; forward = engine.Plan.nonlocal_block)."""

    def __init__(self, dim, dim_inner, pool_size=None, instantiation="softmax", zero_init_final_conv=False,
                 zero_init_final_norm=True, norm_eps=1e-5, norm_momentum=0.1, norm_module=nn.BatchNorm3d):
        super().__init__()
        self.dim, self.dim_inner, self.pool_size, self.instantiation = dim, dim_inner, pool_size, instantiation
        self.use_pool = False if pool_size is None else any((size > 1 for size in pool_size))
        self.conv_theta = nn.Conv3d(dim, dim_inner, kernel_size=1, stride=1, padding=0)
        self.conv_phi = nn.Conv3d(dim, dim_inner, kernel_size=1, stride=1, padding=0)
        self.conv_g = nn.Conv3d(dim, dim_inner, kernel_size=1, stride=1, padding=0)
        self.conv_out = nn.Conv3d(dim_inner, dim, kernel_size=1, stride=1, padding=0)
        self.conv_out.zero_init = zero_init_final_conv
        self.bn = norm_module(num_features=dim, eps=norm_eps, momentum=norm_momentum)
        self.bn.transform_final_bn = zero_init_final_norm
        if self.use_pool:
            self.pool = nn.MaxPool3d(kernel_size=pool_size, stride=pool_size, padding=[0, 0, 0])


class ResStage(_Holder):
    """resnet_helper.py:361-561, Nonlocal blocks after the listed residual blocks included."""

    def __init__(self, dim_in, dim_out, stride, temp_kernel_sizes, num_blocks, dim_inner, num_groups,
                 num_block_temp_kernel, nonlocal_inds, dilation, trans_func_name, stride_1x1, norm_module,
                 nonlocal_group=None, nonlocal_pool=None, instantiation="softmax"):
        super().__init__()
        assert all(num_block_temp_kernel[i] <= num_blocks[i] for i in range(len(temp_kernel_sizes)))
        if trans_func_name != "bottleneck_transform":
            # The reference cannot build "basic_transform" either: ResBlock passes `dilation=` to the transform
            # (resnet_helper.py:336-347) and BasicTransform.__init__ (resnet_helper.py:30-43) has no such parameter ->
            # TypeError at construction.  bottleneck_transform is the only transform its model zoo can instantiate.
            raise NotImplementedError("RESNET.TRANS_FUNC '%s': only bottleneck_transform can be instantiated (the "
                                      "reference's basic_transform raises TypeError at construction)" % trans_func_name)
        self.nonlocal_group = nonlocal_group if nonlocal_group is not None else [1] * len(num_blocks)
        nonlocal_pool = nonlocal_pool if nonlocal_pool is not None else [[1, 2, 2]] * len(num_blocks)
        self.num_blocks = num_blocks
        self.temp_kernel_sizes = [
            (temp_kernel_sizes[i] * num_blocks[i])[: num_block_temp_kernel[i]]
            + [1] * (num_blocks[i] - num_block_temp_kernel[i])
            for i in range(len(temp_kernel_sizes))
        ]
        self.num_pathways = len(num_blocks)
        for p in range(self.num_pathways):
            for i in range(num_blocks[p]):
                blk = ResBlock(dim_in[p] if i == 0 else dim_out[p], dim_out[p], self.temp_kernel_sizes[p][i],
                               stride[p] if i == 0 else 1, dim_inner[p], num_groups[p], stride_1x1, dilation[p],
                               norm_module)
                self.add_module("pathway{}_res{}".format(p, i), blk)
                if i in nonlocal_inds[p]:
                    nln = Nonlocal(dim_out[p], dim_out[p] // 2, nonlocal_pool[p], instantiation=instantiation,
                                   norm_module=norm_module)
                    self.add_module("pathway{}_nonlocal{}".format(p, i), nln)


class FuseFastToSlow(_Holder):
    """video_model_builder.py:93-150: conv kx1x1 stride (alpha,1,1) C->ratio*C -> BN -> ReLU -> cat into slow."""

    def __init__(self, dim_in, fusion_conv_channel_ratio, fusion_kernel, alpha, norm_module, eps=1e-5, bn_mmt=0.1):
        super().__init__()
        self.alpha = alpha
        self.conv_f2s = nn.Conv3d(dim_in, dim_in * fusion_conv_channel_ratio, kernel_size=[fusion_kernel, 1, 1],
                                  stride=[alpha, 1, 1], padding=[fusion_kernel // 2, 0, 0], bias=False)
        self.bn = norm_module(num_features=dim_in * fusion_conv_channel_ratio, eps=eps, momentum=bn_mmt)
        self.relu = nn.ReLU(True)


class SpatialAttention(_Holder):
    """wdf_attention_helper.py:13-54 (position attention; gamma starts at zero)."""

    def __init__(self, channel, reduction=8):
        super().__init__()
        self.input_channel = channel
        self.query_conv = nn.Conv3d(channel, channel // reduction, kernel_size=1)
        self.key_conv = nn.Conv3d(channel, channel // reduction, kernel_size=1)
        self.value_conv = nn.Conv3d(channel, channel, kernel_size=1)
        self.gamma = nn.Parameter(torch.zeros(1))
        self.softmax = nn.Softmax(dim=-1)


class ECA(_Holder):
    """wdf_attention_helper.py:57-91."""

    def __init__(self, channel, k_size=3):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool3d(1)
        self.conv = nn.Conv1d(1, 1, kernel_size=k_size, padding=(k_size - 1) // 2, bias=False)
        self.sigmoid = nn.Sigmoid()


class FuseFastAndSlow(_Holder):
    """CMDA, custom_video_model_builder.py:42-148."""

    def __init__(self, dim_in, alpha, beta_inv, norm_module, eps=1e-5, bn_mmt=0.1, reduction=1):
        super().__init__()
        self.alpha = alpha
        self.downsample_t_of_fast = nn.MaxPool3d(kernel_size=(alpha, 1, 1), stride=(alpha, 1, 1))
        self.attention_channel_f2s = ECA(dim_in[1])
        self.bn_f2s = norm_module(num_features=dim_in[1], eps=eps, momentum=bn_mmt)
        self.relu_f2s = nn.ReLU(True)
        self.downsample_c_of_slow = nn.Conv3d(dim_in[0], dim_in[0] // beta_inv, kernel_size=[1, 1, 1],
                                              stride=[1, 1, 1], bias=False)
        self.attention_spatial_s2f = SpatialAttention(int(dim_in[0] // beta_inv), reduction=reduction)
        self.bn_s2f = norm_module(num_features=int(dim_in[0] // beta_inv), eps=eps, momentum=bn_mmt)
        self.relu_s2f = nn.ReLU(True)
        self.upsample_s2f = nn.Upsample(scale_factor=(alpha, 1, 1), mode="nearest")


class ResNetBasicHead(_Holder):
    """head_helper.py:133-223."""

    def __init__(self, dim_in, num_classes, pool_size, dropout_rate=0.0, act_func="softmax"):
        super().__init__()
        assert len({len(pool_size), len(dim_in)}) == 1, "pathway dimensions are not consistent."
        self.num_pathways = len(pool_size)
        self.pool_size = pool_size
        for p in range(self.num_pathways):
            pool = nn.AdaptiveAvgPool3d((1, 1, 1)) if pool_size[p] is None else nn.AvgPool3d(pool_size[p], stride=1)
            self.add_module("pathway{}_avgpool".format(p), pool)
        if dropout_rate > 0.0:
            self.dropout = nn.Dropout(dropout_rate)
        self.projection = nn.Linear(sum(dim_in), num_classes, bias=True)
        if act_func == "softmax":
            self.act = nn.Softmax(dim=4)
        elif act_func == "sigmoid":
            self.act = nn.Sigmoid()
        else:
            raise NotImplementedError("{} is not supported as an activation function.".format(act_func))
        self.act_func = act_func


class ROIAlign(_Holder):
    """detectron2.layers.ROIAlign (parameter-free): output_size, spatial_scale, sampling_ratio, aligned.  The sampling
    itself is esf_roi_align_max (torchvision roi_align semantics, which detectron2's ROIAlign dispatches to)."""

    def __init__(self, output_size, spatial_scale, sampling_ratio, aligned=True):
        super().__init__()
        self.output_size, self.spatial_scale = output_size, spatial_scale
        self.sampling_ratio, self.aligned = sampling_ratio, aligned


class ResNetRoIHead(_Holder):
    """head_helper.py:12-130 (AVA detection): per pathway a temporal AvgPool3d, RoIAlign and a spatial MaxPool2d over the
    RoIAlign output, then concat -> Linear -> softmax(dim=1) / sigmoid.  One row per box."""

    def __init__(self, dim_in, num_classes, pool_size, resolution, scale_factor, dropout_rate=0.0, act_func="softmax",
                 aligned=True):
        super().__init__()
        assert len({len(pool_size), len(dim_in)}) == 1, "pathway dimensions are not consistent."
        self.num_pathways = len(pool_size)
        for p in range(self.num_pathways):
            self.add_module("s{}_tpool".format(p), nn.AvgPool3d([pool_size[p][0], 1, 1], stride=1))
            self.add_module("s{}_roi".format(p), ROIAlign(resolution[p], spatial_scale=1.0 / scale_factor[p],
                                                         sampling_ratio=0, aligned=aligned))
            self.add_module("s{}_spool".format(p), nn.MaxPool2d(resolution[p], stride=1))
        if dropout_rate > 0.0:
            self.dropout = nn.Dropout(dropout_rate)
        self.projection = nn.Linear(sum(dim_in), num_classes, bias=True)
        if act_func == "softmax":
            self.act = nn.Softmax(dim=1)
        elif act_func == "sigmoid":
            self.act = nn.Sigmoid()
        else:
            raise NotImplementedError("{} is not supported as an activation function.".format(act_func))
        self.act_func = act_func


def init_weights(model, fc_init_std=0.01, zero_init_final_bn=True):
    """utils/weight_init_helper.py:10-43: c2_msra_fill (kaiming normal, fan_out, relu; zero bias) on Conv3d, BN weight
    1 (0 for the last BN of a bottleneck when zero_init_final_bn), BN bias 0, Linear N(0, fc_init_std) / zero bias.
    Conv1d (ECA) keeps its constructor init, as in the reference."""
    for m in model.modules():
        if isinstance(m, nn.Conv3d):
            nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.BatchNorm3d):
            zero = getattr(m, "transform_final_bn", False) and zero_init_final_bn
            if m.weight is not None:
                m.weight.data.fill_(0.0 if zero else 1.0)
            if m.bias is not None:
                m.bias.data.zero_()
        if isinstance(m, nn.Linear):
            m.weight.data.normal_(mean=0.0, std=fc_init_std)
            m.bias.data.zero_()


# --------------------------------------------------------------------------------------------- model base
class _PlannedModel(nn.Module):
    """Shared forward machinery: shape-keyed launch plans, weight-version tracking, CUDA-graph replay."""

    num_pathways = 2
    supports_fp32 = False     # cfg.ESF.PRECISION = "fp32" (engine_fp32.PrecisePlan): every classification model here
    enable_detection = False  # cfg.DETECTION.ENABLE: ResNetRoIHead, forward(x, bboxes) returns one row per box

    def _init_runtime(self, cfg):
        self._cfg = cfg
        self._plans = collections.OrderedDict()     # (shapes, device) -> (weights stamp, Plan), least recently used first
        esf = cfg.get("ESF", {}) if hasattr(cfg, "get") else {}
        self._use_graph = bool(esf.get("CUDA_GRAPH", True))
        # live plans kept per model: the activation arena of a plan is large (25 GB at batch 64), but a test loader
        # alternates between the full batch and a short last one, and the demo between window and batch shapes
        self._max_plans = max(1, int(esf.get("MAX_PLANS", 2)))
        # batch capacity (0: off): one plan family per per-clip input shape serves every batch of up to MAX_BATCH rows
        self._max_batch = int(esf.get("MAX_BATCH", 0) or 0)
        if self._max_batch < 0:
            raise ValueError("cfg.ESF.MAX_BATCH must be >= 0 (0: off), got %d" % self._max_batch)

    def _weights_stamp(self):
        """Identity of the weights a plan was compiled from: (storage address, version counter) of every parameter
        and buffer.  In-place edits through autograd-visible ops and load_state_dict bump the version; edits through
        `.data` / `.detach()` views do NOT (PyTorch gives them no counter) -- call invalidate_plans() after those
        (load_state_dict / .to() / .cuda() do it themselves)."""
        return hash(tuple((t.data_ptr(), t._version) for t in itertools.chain(self.parameters(), self.buffers())))

    def invalidate_plans(self):
        self._plans.clear()

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate_plans()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        if hasattr(self, "_plans"):
            self.invalidate_plans()
        return out

    def _get_plan(self, shapes, device):
        """The plan for input `shapes` on `device`, compiled on first use.  With cfg.ESF.MAX_BATCH = N the key leaves
        out the batch rows (dim 0): the first call compiles the family's capacity plan at N rows, a call with b < N rows
        gets the family's variant for b (engine.Family), and b > N raises EsfError before anything is launched."""
        shapes = [tuple(int(n) for n in s) for s in shapes]
        cap = self._max_batch
        if cap and shapes[0][0] > cap:
            raise rt.EsfError("a batch of %d rows exceeds cfg.ESF.MAX_BATCH = %d, the capacity of the compiled plans"
                              % (shapes[0][0], cap))
        key = (tuple(s[1:] if cap else s for s in shapes), str(device))
        stamp = self._weights_stamp()
        ent = self._plans.get(key)
        if ent is not None and ent[0] == stamp:
            self._plans.move_to_end(key)
            return self._variant(ent[1], shapes) if cap else ent[1]
        self._check_roi_time_axis(shapes)            # before any cached plan is evicted for this shape
        if ent is not None or any(st != stamp for st, _ in self._plans.values()):
            self._plans.clear()                      # the weights changed: every compiled plan is stale
        prec = "fp16"
        if hasattr(self._cfg, "get") and self._cfg.get("ESF") is not None:
            prec = str(self._cfg.ESF.get("PRECISION", "fp16"))
        if prec == "fp32" and self.enable_detection:
            raise NotImplementedError("ESF.PRECISION = 'fp32' does not cover the detection head (DETECTION.ENABLE); run "
                                      "detection models with 'fp16' / 'bf16'")
        while len(self._plans) >= self._max_plans:
            self._plans.popitem(last=False)          # frees the arena of the least recently used shape
        if cap:
            plan = self._compile_plan([(cap,) + s[1:] for s in shapes], device, prec, Family())
        else:
            plan = self._compile_plan(shapes, device, prec)
        self._plans[key] = (stamp, plan)
        return self._variant(plan, shapes) if cap else plan

    def _variant(self, plan, shapes):
        """The plan of the family of capacity plan `plan` for `shapes` (their batch rows at most the capacity)."""
        b = shapes[0][0]
        if b == plan.inputs[0].shape[0]:
            return plan
        if b not in plan.variants:
            plan.variants[b] = self._compile_plan(shapes, plan.device, plan.precision, plan.family)
        return plan.variants[b]

    def _compile_plan(self, shapes, device, prec, family=None):
        """Compile a plan for input `shapes` at precision `prec`, as a member of `family` when given."""
        with torch.cuda.device(device):
            if prec == "fp32":
                if not self.supports_fp32:
                    raise NotImplementedError("ESF.PRECISION = 'fp32' (FP32-accurate plan) covers the ResNet based "
                                              "models; %s runs with 'fp16' / 'bf16'" % type(self).__name__)
                from .engine_fp32 import PrecisePlan
                plan = PrecisePlan(device, family=family)
            else:
                plan = Plan(device, precision=prec, family=family)
            plan.inputs = [plan.alloc(s, torch.float32) for s in shapes]
            with torch.no_grad():
                self._compile(plan)
            if family is not None:
                plan.end_compile()
            if self._use_graph:
                plan.capture()
        return plan

    def input_buffers(self, shapes, device=None):
        """Plan-owned static input tensors for `shapes`; filling these (e.g. as the target of the H2D copy) and then
        calling forward() on them skips the device-to-device staging copy."""
        device = device or next(self.parameters()).device
        return self._get_plan(shapes, device).inputs

    def forward(self, x, bboxes=None):
        assert len(x) == self.num_pathways, "Input tensor does not contain {} pathway".format(self.num_pathways)
        if self.training:
            raise NotImplementedError("efficient_slowfast_b200 implements the eval-mode forward path only; call "
                                      ".eval() (training / autograd is outside the accelerated hot path)")
        dev = x[0].device
        boxes = self._boxes(bboxes, x[0].shape[0], dev)
        if dev.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got tensors on %s -- there is no CPU fallback"
                              % dev)
        if x[0].shape[0] == 0 or (boxes is not None and boxes.shape[0] == 0):
            # an empty batch is an empty result (nn.Conv3d / nn.Linear of the reference agree); so is an empty box list
            return self._empty(dev)
        plan = self._get_plan([tuple(t.shape) for t in x], dev)
        # FP32 contiguous clips are read in place by the stem kernels (launched outside the CUDA graph); anything else
        # (other dtype / strides) is first converted into the plan-owned input buffers
        direct = all(t.dtype == torch.float32 and t.is_contiguous() and t.data_ptr() % 16 == 0 for t in x)
        with torch.cuda.device(dev):     # launches go to the tensors' device and ITS current stream
            if not direct:
                for src, dst in zip(x, plan.inputs):
                    if src.data_ptr() != dst.data_ptr():
                        dst.copy_(src, non_blocking=True)
            out = plan.run(list(x) if direct else None)
            return self._finish(plan, out, boxes)

    def forward_fast(self, fast, bboxes=None):
        """Same result as `forward(pack_pathway_output(cfg, fast))`: the loader's pack_pathway_output
        (SlowFast/slowfast/datasets/utils.py:93-102) makes the slow clip out of the
        `linspace(0, T-1, T // ALPHA).long()` frames of the fast clip, i.e. the same pixels a second time (20 % of the
        host-to-device bytes of a batch).  Here only the fast clip (B, C, T, H, W) FP32 is given; the slow pathway's
        stem packs its rows straight out of those frames (esf_stem_pack_gather), so the slow clip is neither uploaded
        nor materialised.  Stems without the packed-row route gather on the device into the plan's slow input."""
        if self.num_pathways != 2:
            raise rt.EsfError("forward_fast is for the two-pathway models")
        if self.training:
            raise NotImplementedError("eval-mode forward path only")
        dev = fast.device
        boxes = self._boxes(bboxes, fast.shape[0], dev)
        if dev.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got tensors on %s -- there is no CPU fallback"
                              % dev)
        if fast.dtype != torch.float32 or fast.dim() != 5 or not fast.is_contiguous() or fast.data_ptr() % 16:
            raise rt.EsfError("forward_fast expects a contiguous FP32 clip (B, C, T, H, W)")
        B, C, T, H, W = fast.shape
        if B == 0 or (boxes is not None and boxes.shape[0] == 0):
            return self._empty(dev)
        alpha = self._cfg.SLOWFAST.ALPHA
        plan = self._get_plan([(B, C, T // alpha, H, W), (B, C, T, H, W)], dev)
        idx = getattr(plan.shared, "slow_index", None)
        if idx is None:
            idx = plan.shared.slow_index = torch.linspace(0, T - 1, T // alpha).long().to(torch.int32).to(dev)
        with torch.cuda.device(dev):
            if plan.inputs[0].data_ptr() in plan.stem_routes:
                out = plan.run([None, fast], gather={0: (fast, idx)})
            else:
                torch.index_select(fast, 2, idx.long(), out=plan.inputs[0])
                out = plan.run([None, fast])
            return self._finish(plan, out, boxes)

    def frame_shapes(self, frames_shape):
        """[slow, fast] (or [single]) clip shapes that pack_pathway_output (datasets/utils.py:73-112) makes of uint8
        frames (B, T, H, W, C)."""
        B, T, H, W, C = frames_shape
        if self.num_pathways == 1:
            return [(B, C, T, H, W)]
        return [(B, C, T // self._cfg.SLOWFAST.ALPHA, H, W), (B, C, T, H, W)]

    def forward_frames(self, frames, bboxes=None, frame_index=None, crop_size=None, spatial_idx=None):
        """Same result as `forward(pack_pathway_output(cfg, tensor_normalize(frames, MEAN, STD).permute(...)))` of the
        reference's loader chain, from the decoder's uint8 frames (B, T, H, W, C) on the device: normalisation,
        layout change and the slow-pathway frame gather run inside the stem-pack kernel (frames.py).

        Test-time spatial sampling: with `spatial_idx` (an int or a sequence of V values from {0, 1, 2}) the frames are
        at decode size and every clip also goes through the reference's test-mode `spatial_sampling` (short side
        resized to `crop_size`, default cfg.DATA.TEST_CROP_SIZE, then `uniform_crop` at each index) on the device.  The
        result has B * V rows, row b * V + v being clip b at view v (the order of the test loader's clip numbering).
        `crop_size` alone means spatial_idx 1 (TEST.NUM_SPATIAL_CROPS = 1).

        Mixed decode sizes: `frames` may also be a list or tuple of B contiguous uint8 clips (T, H_b, W_b, C) on one
        device, of one T and C.  A list always means test-time spatial sampling (same defaults); every clip is resized
        and cropped on its own, as the reference's loader does before collating.  The plan is that of a stacked batch
        of B clips, so batches of any mix of sizes share it, and a list of clips of one size gives the stacked result
        bit for bit."""
        from . import frames as esf_frames
        if self.training:
            raise NotImplementedError("eval-mode forward path only")
        if isinstance(frames, (list, tuple)):
            return self._forward_clip_list(list(frames), bboxes, frame_index, crop_size, spatial_idx)
        crop = crop_size is not None or spatial_idx is not None
        if crop:
            if bboxes is not None:
                raise ValueError("forward_frames: bboxes together with spatial_idx is not supported (the boxes would "
                                 "need the crop's transform)")
            views = esf_frames.spatial_views(1 if spatial_idx is None else spatial_idx)
            crop_size = int(self._cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
            if frames.dim() != 5:
                raise rt.EsfError("forward_frames expects contiguous uint8 frames (B, T, H, W, C)")
            shapes = esf_frames.view_shapes(tuple(frames.shape), crop_size, views,
                                            self._cfg.SLOWFAST.ALPHA if self.num_pathways > 1 else None)
        boxes = self._boxes(bboxes, frames.shape[0] if frames.dim() else 0, frames.device)
        if frames.device.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got frames on %s -- there is no CPU fallback"
                              % frames.device)
        if frames.dtype != torch.uint8 or frames.dim() != 5 or not frames.is_contiguous():
            raise rt.EsfError("forward_frames expects contiguous uint8 frames (B, T, H, W, C)")
        dev = frames.device
        alpha = self._cfg.SLOWFAST.ALPHA if self.num_pathways > 1 else 1
        if not crop:
            shapes = self.frame_shapes(tuple(frames.shape))
        if frames.shape[0] == 0 or (boxes is not None and boxes.shape[0] == 0):
            return self._empty(dev)
        if frame_index is not None:     # explicit source frame of every pathway frame (frames may be a ring buffer)
            assert len(frame_index) == self.num_pathways
            shapes = [tuple(sh[:2]) + (int(ix.numel()),) + tuple(sh[3:]) for sh, ix in zip(shapes, frame_index)]
        plan, fin = self._frame_plan(shapes, dev, frames.shape[4])
        tabs = fin.crop(frames.shape[2], frames.shape[3], crop_size, views) if crop else None
        with torch.cuda.device(dev):
            out = plan.run_frames(lambda: esf_frames.launch_frames(plan, fin, frames, alpha, frame_index, tabs))
            return self._finish(plan, out, boxes)

    def _frame_plan(self, shapes, dev, channels):
        """The plan for `shapes` and its FrameInput (frames.py) for frames of `channels` channels."""
        from . import frames as esf_frames
        plan = self._get_plan(shapes, dev)
        fin = getattr(plan.shared, "frame_input", None)
        if fin is None:
            fin = plan.shared.frame_input = esf_frames.FrameInput(self._cfg, dev, plan.adt, channels=channels)
        return plan, fin

    def _forward_clip_list(self, clips, bboxes, frame_index, crop_size, spatial_idx):
        """forward_frames on a list of clips of mixed decode sizes: every argument is checked before anything runs."""
        from . import frames as esf_frames
        if bboxes is not None or frame_index is not None:
            raise ValueError("forward_frames: a list of clips takes neither bboxes nor frame_index (the boxes would need "
                             "each crop's transform)")
        views = esf_frames.spatial_views(1 if spatial_idx is None else spatial_idx)
        crop_size = int(self._cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
        if not clips:
            return self._empty(next(self.parameters()).device)
        sizes = esf_frames.check_clips(clips)
        shapes = esf_frames.view_shapes(sizes, crop_size, views,
                                        self._cfg.SLOWFAST.ALPHA if self.num_pathways > 1 else None)
        dev = clips[0].device
        if dev.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got frames on %s -- there is no CPU fallback"
                              % dev)
        alpha = self._cfg.SLOWFAST.ALPHA if self.num_pathways > 1 else 1
        plan, fin = self._frame_plan(shapes, dev, sizes[0][3])
        batch = esf_frames.ClipList(clips, [fin.crop(H, W, crop_size, views) for _, H, W, _ in sizes])
        with torch.cuda.device(dev):
            out = plan.run_frames(lambda: esf_frames.launch_clip_list(plan, fin, batch, alpha))
            return self._finish(plan, out, None)

    def forward_videos(self, videos, fps=None, num_clips=None, spatial_idx=None, crop_size=None, bboxes=None):
        """The reference's whole test protocol from decoded videos: every video is tested as `num_clips` temporal clips
        (default cfg.TEST.NUM_ENSEMBLE_VIEWS) x V crops (default the test loader's views for cfg.TEST.NUM_SPATIAL_CROPS:
        (0, 1, 2) for 3, (1,) for 1).  Temporal clip j of a video is what the reference's decoder samples when it has
        decoded the whole video (datasets/decoder.py: get_start_end_idx(N, clip_size, j, num_clips) and
        temporal_sampling, clip_size = SAMPLING_RATE * NUM_FRAMES / TARGET_FPS * fps); each clip then goes through the
        loader's normalisation, short-side resize to `crop_size` (default cfg.DATA.TEST_CROP_SIZE), uniform crops and
        pack_pathway_output, as in forward_frames.  The pyav branch that seeks to a per-clip timestamp window (whose
        frames depend on the container's keyframes) is not covered.

        `videos`: list of contiguous uint8 videos (N_v, H_v, W_v, C) on one CUDA device, of any length and size, one
        C.  `fps`: a number or one per video (default cfg.DATA.TARGET_FPS).  Each video is read in place; only the
        frame tables (a few KB) are uploaded.  The result has len(videos) * num_clips * V rows, row
        (v * num_clips + j) * V + s being video v, temporal clip j, crop s: the order of the test loader's clip
        numbering, so TestMeter.update_stats takes the rows with clip ids video_idx * num_clips * V + row.  The plan
        is that of forward_frames on a stacked batch of len(videos) * num_clips clips, so both routes share it."""
        from . import frames as esf_frames
        if self.training:
            raise NotImplementedError("eval-mode forward path only")
        if bboxes is not None:
            raise ValueError("forward_videos takes no bboxes (the boxes would need each view's transform)")
        if not isinstance(videos, (list, tuple)):
            raise ValueError("forward_videos takes a list of videos (N, H, W, C), got %s" % type(videos).__name__)
        cfg = self._cfg
        target_fps = cfg.DATA.get("TARGET_FPS", 30) if hasattr(cfg.DATA, "get") else cfg.DATA.TARGET_FPS
        num_clips = cfg.TEST.NUM_ENSEMBLE_VIEWS if num_clips is None else num_clips
        views = esf_frames.spatial_views(esf_frames.ensemble_spatial_views(cfg.TEST.NUM_SPATIAL_CROPS)
                                         if spatial_idx is None else spatial_idx)
        crop_size = int(cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
        sizes, rates = esf_frames.check_videos(list(videos), target_fps if fps is None else fps, num_clips)
        if not sizes:
            return self._empty(next(self.parameters()).device)
        two = self.num_pathways > 1
        T = int(cfg.DATA.NUM_FRAMES)
        shapes = esf_frames.view_shapes([(T, H, W, C) for _, H, W, C in sizes for _ in range(num_clips)], crop_size,
                                        views, cfg.SLOWFAST.ALPHA if two else None)
        dev = videos[0].device
        if dev.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got videos on %s -- there is no CPU fallback"
                              % dev)
        plan, fin = self._frame_plan(shapes, dev, sizes[0][3])
        crops = [fin.crop(H, W, crop_size, views) for _, H, W, _ in sizes]
        tables = [fin.video_tables(N, f, T, int(cfg.DATA.SAMPLING_RATE), target_fps, int(num_clips),
                                   cfg.SLOWFAST.ALPHA if two else None) for (N, _, _, _), f in zip(sizes, rates)]
        batch = esf_frames.VideoList(list(videos), crops, tables, int(num_clips))
        with torch.cuda.device(dev):
            out = plan.run_frames(lambda: esf_frames.launch_video_list(plan, fin, batch))
            return self._finish(plan, out, None)

    def forward_ava_frames(self, frames, boxes, crop_size=None, return_boxes=False):
        """AVA detection from the decoder's uint8 frames: the same result as `forward(clips, bboxes)` on what the test
        split of the reference's AVA loader makes of them (datasets/ava_dataset.py _images_and_boxes_preprocessing,
        PyTorch backend): `frames / 255`, the boxes times (W, H) and clipped to the frame, a bilinear short-side resize to
        `crop_size` (default cfg.DATA.TEST_CROP_SIZE) with the boxes scaled alike and no crop, color_normalization with
        DATA.MEAN / DATA.STD, the BGR -> RGB swap unless cfg.AVA.BGR, the boxes clipped to crop_size x crop_size, and
        pack_pathway_output.  All of it runs on the device (csrc/esf_crop.cu): frames and boxes are read in place.

        `frames`: contiguous uint8 (B, T, H, W, C) on a CUDA device, the loader's sampled frames at decode size.
        `boxes`: floating (K, 5) rows [batch index, x1, y1, x2, y2] with coordinates in [0, 1] (the annotation format), on
        the host (checked before anything runs) or on the device (read by the kernel, no synchronisation); FP64 boxes
        keep the loader's FP64 arithmetic exactly.  Returns the (K, NUM_CLASSES) scores, and with `return_boxes` also
        the transformed FP32 (K, 5) boxes in resized-frame pixels.  The plan is that of `forward(clips, bboxes)` on clips
        of the resized size, and any number of boxes reuses its graph.  AVA.TEST_FORCE_FLIP is not covered."""
        from . import frames as esf_frames
        if self.training:
            raise NotImplementedError("eval-mode forward path only")
        if not self.enable_detection:
            raise NotImplementedError("forward_ava_frames needs a detection model (cfg.DETECTION.ENABLE, ResNetRoIHead)")
        cfg = self._cfg
        ava = cfg.get("AVA", None) if hasattr(cfg, "get") else None
        if ava is not None and hasattr(ava, "get") and bool(ava.get("TEST_FORCE_FLIP", False)):
            raise NotImplementedError("AVA.TEST_FORCE_FLIP (the test branch's horizontal flip) is not covered by "
                                      "forward_ava_frames")
        B, T, H, W, C = esf_frames.check_ava_frames(frames)
        b = esf_frames.check_ava_boxes(boxes, B)
        S = int(cfg.DATA.TEST_CROP_SIZE if crop_size is None else crop_size)
        if S < 1:
            raise ValueError("crop_size must be >= 1, got %d" % S)
        dev = frames.device
        if dev.type != "cuda":
            raise rt.EsfError("the forward path is CUDA-only (sm_100a); got frames on %s -- there is no CPU fallback"
                              % dev)
        Hr, Wr = esf_frames.resized_size(H, W, S)
        shapes = self.frame_shapes((B, T, Hr, Wr, C))
        K = b.shape[0]
        if B == 0 or K == 0:
            out = self._empty(dev)
            return (out, torch.empty((0, 5), dtype=torch.float32, device=dev)) if return_boxes else out
        alpha = cfg.SLOWFAST.ALPHA if self.num_pathways > 1 else 1
        plan, fin = self._frame_plan(shapes, dev, C)
        state = fin.ava(cfg)
        tabs = fin.crop(H, W, S, ())
        with torch.cuda.device(dev):
            if b.device.type == "cpu":   # staged through pinned memory, as forward's boxes: no wait for earlier work
                staged = torch.empty(b.shape, dtype=b.dtype, pin_memory=True)
                staged.copy_(b)
                b = staged.to(dev, non_blocking=True)
            elif b.device != dev:
                b = b.to(dev)
            px = torch.empty((K, 5), dtype=torch.float32, device=dev)
            esf_frames.launch_ava_boxes(b, tabs, px)
            out = plan.run_frames(lambda: esf_frames.launch_ava(plan, fin, state, frames, tabs, alpha))
            out = self._finish(plan, out, px)
        return (out, px) if return_boxes else out

    def _empty(self, dev):
        return torch.empty((0, int(self._cfg.MODEL.NUM_CLASSES)), dtype=torch.float32, device=dev)

    def _check_roi_time_axis(self, shapes):
        """ResNetRoIHead's temporal AvgPool3d([t, 1, 1], stride 1) must leave one frame of every pathway's res5 output:
        the reference asserts `out.shape[2] == 1` after it (head_helper.py) and AvgPool3d itself rejects t > T.  The
        trunk keeps the time axis except for the max-pool after res2 (kernel = stride = pathway{p}_pool)."""
        if not self.enable_detection:
            return
        for p, shape in enumerate(shapes):
            k = int(getattr(self, "pathway%d_pool" % p).kernel_size[0])
            T = (int(shape[2]) - k) // k + 1
            kt = int(getattr(self.head, "s%d_tpool" % p).kernel_size[0])
            if kt > T:
                raise RuntimeError("head temporal AvgPool3d kernel %d is larger than the %d res5 frames of pathway %d"
                                   % (kt, T, p))
            if T - kt + 1 != 1:
                raise AssertionError("pathway %d: the head's temporal pool (kernel %d) leaves %d frames of %d, the "
                                     "reference's ResNetRoIHead asserts 1" % (p, kt, T - kt + 1, T))

    def _boxes(self, bboxes, batch, dev):
        """Detection models: `bboxes` (K, 5) rows [batch index, x1, y1, x2, y2] in input pixels, as one contiguous FP32
        tensor on `dev` (a single copy).  Host boxes are checked before anything is launched: shape, and batch indices
        in [0, batch).  Device boxes are only shape-checked (reading them would synchronise); there the kernel clamps the
        batch index and writes NaN rows for non-finite boxes.  Classification models: None, and `bboxes` must be None."""
        if not self.enable_detection:
            if bboxes is not None:
                raise NotImplementedError("bboxes given to a classification model; detection needs a model built with "
                                          "cfg.DETECTION.ENABLE (ResNetRoIHead)")
            return None
        if bboxes is None:
            raise ValueError("detection model (cfg.DETECTION.ENABLE): forward needs bboxes, a (K, 5) tensor of "
                             "[batch index, x1, y1, x2, y2]")
        if (not torch.is_tensor(bboxes) or not bboxes.is_floating_point() or bboxes.dim() != 2
                or bboxes.shape[1] != 5):
            raise ValueError("bboxes must be a floating-point (K, 5) tensor of [batch index, x1, y1, x2, y2]; got %s"
                             % ((tuple(bboxes.shape), bboxes.dtype) if torch.is_tensor(bboxes) else type(bboxes).__name__,))
        if bboxes.device.type == "cpu":
            b = bboxes.detach().to(torch.float32).contiguous()
            idx = b[:, 0]
            bad = ~((idx >= 0) & (idx < batch))
            if bool(bad.any()):
                raise ValueError("bboxes[:, 0] must be batch indices in [0, %d); got %s"
                                 % (batch, idx[bad][:4].tolist()))
            if dev.type != "cuda":
                return b
            # staged through pinned memory: the copy is queued on the stream instead of waiting for earlier work.  The
            # host caching allocator keeps the staging block until the copy has run, although the tensor dies here.
            staged = torch.empty(b.shape, dtype=torch.float32, pin_memory=True)
            staged.copy_(b)
            with torch.cuda.device(dev):
                return staged.to(dev, non_blocking=True)
        return bboxes.detach().to(device=dev, dtype=torch.float32).contiguous()

    @staticmethod
    def _finish(plan, out, boxes):
        """The caller's copy of the result; detection plans first run their box-dependent launches (Plan.run_boxes)."""
        if boxes is not None:
            out = plan.run_boxes(boxes)
        return out.clone()

    def _emit_fuse(self, plan, fuse, cur):
        (sbuf, soff, cs), (fbuf, foff, cf) = cur
        x_s = sbuf[..., soff:soff + cs]
        x_f = fbuf[..., foff:foff + cf]
        if isinstance(fuse, FuseFastAndSlow):
            # fast -> slow: written behind x_s;  slow -> fast: written in front of x_f.  Both read only stage outputs.
            plan.eca_fuse(x_f, sbuf[..., cs:cs + cf], fuse.alpha, fuse.attention_channel_f2s.conv.weight, fuse.bn_f2s)
            d = fuse.downsample_c_of_slow.out_channels
            plan.position_attention(x_s, fbuf[..., 0:d], fuse.alpha, fuse.downsample_c_of_slow.weight,
                                    fuse.attention_spatial_s2f, fuse.bn_s2f)
        else:
            conv = fuse.conv_f2s
            w, b = plan.once(fold_conv_bn, conv.weight, None, fuse.bn)
            plan.conv(x_f, sbuf[..., cs:cs + conv.out_channels], w, b, stride=tuple(conv.stride),
                      padding=tuple(conv.padding), act=rt.ACT_RELU)

    def debug_buffers(self):
        """name -> channels-last BF16 activation tensors of the live plan (tests only)."""
        for _, plan in reversed(self._plans.values()):    # most recently used
            return plan.buffers
        return {}


def _stage_dims(cfg):
    w = cfg.RESNET.WIDTH_PER_GROUP
    return [w * 4, w * 8, w * 16, w * 32]


class _TwoStreamResNet(_PlannedModel):
    """Common structure of SlowFast and SlowFastDualAttention: stem, 4 residual stages, a fusion module after the
    stem and after res2..res4, identity pathway pools, basic head."""

    supports_fp32 = True

    def _build(self, cfg, dual_attention):
        assert cfg.MODEL.ARCH in _POOL1.keys()
        pool_size = _POOL1[cfg.MODEL.ARCH]
        assert len({len(pool_size), self.num_pathways}) == 1
        assert cfg.RESNET.DEPTH in _MODEL_STAGE_DEPTH.keys()
        if cfg.DETECTION.ENABLE and dual_attention:
            raise NotImplementedError("DETECTION.ENABLE with SlowFastDualAttention: the fork's detection builder for this "
                                      "model could not be checked; detection runs on SlowFast and ResNet")
        self.norm_module = get_norm(cfg)
        self.enable_detection = bool(cfg.DETECTION.ENABLE)
        self.dual_attention = dual_attention
        depths = _MODEL_STAGE_DEPTH[cfg.RESNET.DEPTH]
        num_groups = cfg.RESNET.NUM_GROUPS
        wpg = cfg.RESNET.WIDTH_PER_GROUP
        dim_inner = num_groups * wpg
        beta = cfg.SLOWFAST.BETA_INV
        alpha = cfg.SLOWFAST.ALPHA
        if dual_attention:
            out_dim_ratio = beta                                                # custom_video_model_builder.py:213
        else:
            out_dim_ratio = beta // cfg.SLOWFAST.FUSION_CONV_CHANNEL_RATIO      # video_model_builder.py:199-201
        tk = _TEMPORAL_KERNEL_BASIS[cfg.MODEL.ARCH]

        def fuse(c_slow):
            if dual_attention:
                return FuseFastAndSlow([c_slow, c_slow // beta], alpha, beta, self.norm_module, reduction=1)
            return FuseFastToSlow(c_slow // beta, cfg.SLOWFAST.FUSION_CONV_CHANNEL_RATIO,
                                  cfg.SLOWFAST.FUSION_KERNEL_SZ, alpha, self.norm_module)

        self.s1 = VideoModelStem(
            dim_in=cfg.DATA.INPUT_CHANNEL_NUM, dim_out=[wpg, wpg // beta],
            kernel=[tk[0][0] + [7, 7], tk[0][1] + [7, 7]], stride=[[1, 2, 2]] * 2,
            padding=[[tk[0][0][0] // 2, 3, 3], [tk[0][1][0] // 2, 3, 3]], norm_module=self.norm_module)
        self.s1_fuse = fuse(wpg)
        c_prev = wpg
        for i, name in enumerate(("s2", "s3", "s4", "s5")):
            c_out = wpg * 4 * (2 ** i)
            fast_in = c_prev // beta + (c_prev // out_dim_ratio if dual_attention else 0)
            stage = ResStage(
                dim_in=[c_prev + c_prev // out_dim_ratio, fast_in], dim_out=[c_out, c_out // beta],
                dim_inner=[dim_inner * (2 ** i), dim_inner * (2 ** i) // beta], temp_kernel_sizes=tk[i + 1],
                stride=cfg.RESNET.SPATIAL_STRIDES[i], num_blocks=[depths[i]] * 2, num_groups=[num_groups] * 2,
                num_block_temp_kernel=cfg.RESNET.NUM_BLOCK_TEMP_KERNEL[i], nonlocal_inds=cfg.NONLOCAL.LOCATION[i], nonlocal_group=cfg.NONLOCAL.GROUP[i],
                nonlocal_pool=cfg.NONLOCAL.POOL[i], instantiation=cfg.NONLOCAL.INSTANTIATION,
                dilation=cfg.RESNET.SPATIAL_DILATIONS[i], trans_func_name=cfg.RESNET.TRANS_FUNC,
                stride_1x1=cfg.RESNET.STRIDE_1X1, norm_module=self.norm_module)
            setattr(self, name, stage)
            if name != "s5":
                setattr(self, name + "_fuse", fuse(c_out))
            if name == "s2":
                for p in range(self.num_pathways):
                    self.add_module("pathway{}_pool".format(p),
                                    nn.MaxPool3d(kernel_size=pool_size[p], stride=pool_size[p], padding=[0, 0, 0]))
            c_prev = c_out
        if self.enable_detection:      # video_model_builder.py: ResNetRoIHead branch of _construct_network
            R = cfg.DETECTION.ROI_XFORM_RESOLUTION
            self.head = ResNetRoIHead(
                dim_in=[wpg * 32, wpg * 32 // beta], num_classes=cfg.MODEL.NUM_CLASSES,
                pool_size=[[cfg.DATA.NUM_FRAMES // alpha // pool_size[0][0], 1, 1],
                           [cfg.DATA.NUM_FRAMES // pool_size[1][0], 1, 1]],
                resolution=[[R] * 2] * 2, scale_factor=[cfg.DETECTION.SPATIAL_SCALE_FACTOR] * 2,
                dropout_rate=cfg.MODEL.DROPOUT_RATE, act_func=cfg.MODEL.HEAD_ACT, aligned=cfg.DETECTION.ALIGNED)
        else:
            if cfg.MULTIGRID.SHORT_CYCLE:
                head_pool = [None, None]
            else:
                c = cfg.DATA.CROP_SIZE // 32
                head_pool = [
                    [cfg.DATA.NUM_FRAMES // alpha // pool_size[0][0], c // pool_size[0][1], c // pool_size[0][2]],
                    [cfg.DATA.NUM_FRAMES // pool_size[1][0], c // pool_size[1][1], c // pool_size[1][2]],
                ]
            self.head = ResNetBasicHead(dim_in=[wpg * 32, wpg * 32 // beta], num_classes=cfg.MODEL.NUM_CLASSES,
                                        pool_size=head_pool, dropout_rate=cfg.MODEL.DROPOUT_RATE,
                                        act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    # ------------------------------------------------------------------------------------------ plan
    def _compile(self, plan):
        cfg = self._cfg
        alpha, beta = cfg.SLOWFAST.ALPHA, cfg.SLOWFAST.BETA_INV
        xs_in = plan.inputs
        B = xs_in[0].shape[0]
        assert xs_in[1].shape[2] == xs_in[0].shape[2] * alpha, \
            "fast pathway must have ALPHA x the frames of the slow pathway"
        wpg = cfg.RESNET.WIDTH_PER_GROUP
        c_fast = wpg // beta
        dual = self.dual_attention
        ratio = cfg.SLOWFAST.FUSION_CONV_CHANNEL_RATIO

        def fused_channels(c_slow):
            """channel widths of the [slow, fast] buffers that hold a stage output plus what the fusion appends."""
            cf = c_slow // beta
            if dual:
                return c_slow + cf, cf + cf
            return c_slow + ratio * cf, cf

        def conv_out(n, k, s, p, d=1):
            return (n + 2 * p - d * (k - 1) - 1) // s + 1

        # ---- stem: conv+BN+ReLU (direct, FP32 clip in) then max-pool into the first concat buffers
        cs_tot, cf_tot = fused_channels(wpg)
        cur = []
        for pw in range(2):
            stem = getattr(self.s1, "pathway{}_stem".format(pw))
            x = xs_in[pw]
            _, _, T, H, W = x.shape
            k, s, p = stem.kernel, stem.stride, stem.padding
            To, Ho, Wo = conv_out(T, k[0], s[0], p[0]), conv_out(H, k[1], s[1], p[1]), conv_out(W, k[2], s[2], p[2])
            cout = stem.conv.out_channels
            y = plan.act(B, To, Ho, Wo, cout)
            w, b = plan.once(fold_conv_bn, stem.conv.weight, None, stem.bn)
            plan.stem(x, y, w, b, tuple(s), tuple(p), act=rt.ACT_RELU)
            Hp, Wp = conv_out(Ho, 3, 2, 1), conv_out(Wo, 3, 2, 1)
            buf = plan.act(B, To, Hp, Wp, cs_tot if pw == 0 else cf_tot, name="s1_cat%d" % pw)
            # slow: [x_s | from_fast]; fast (dual attention): [from_slow | x_f]
            off = 0 if (pw == 0 or not dual) else c_fast
            plan.pool(y, buf[..., off:off + cout], (1, 3, 3), (1, 2, 2), (0, 1, 1))
            cur.append((buf, off, cout))
        self._emit_fuse(plan, self.s1_fuse, cur)

        # ---- residual stages
        c_prev = wpg
        for i, name in enumerate(("s2", "s3", "s4", "s5")):
            stage = getattr(self, name)
            c_out = wpg * 4 * (2 ** i)
            last = name == "s5"
            nxt = []
            for pw in range(2):
                buf_in, _, _ = cur[pw]
                x = buf_in                      # the stage consumes the whole concat buffer
                co = c_out if pw == 0 else c_out // beta
                stride = cfg.RESNET.SPATIAL_STRIDES[i][pw]
                dil = cfg.RESNET.SPATIAL_DILATIONS[i][pw]
                _, T, H, W, _ = x.shape
                Ho, Wo = conv_out(H, 1, stride, 0), conv_out(W, 1, stride, 0)
                if last:
                    tot, off = co, 0
                else:
                    tots = fused_channels(c_out)
                    tot = tots[pw]
                    off = 0 if (pw == 0 or not dual) else c_out // beta
                dst = plan.act(B, T, Ho, Wo, tot, name="%s_cat%d" % (name, pw))
                self._emit_stage_pathway(plan, stage, pw, x, dst[..., off:off + co], stride, dil)
                nxt.append((dst, off, co))
            cur = nxt
            if not last:
                self._emit_fuse(plan, getattr(self, name + "_fuse"), cur)
            c_prev = c_out

        # ---- head
        xs = [c[0] for c in cur]
        act = {"softmax": rt.HEAD_SOFTMAX, "sigmoid": rt.HEAD_SIGMOID}[self.head.act_func]
        if self.enable_detection:
            return self._emit_roi_head(plan, xs, act)
        self._emit_head(plan, xs, act)

    def _emit_head(self, plan, xs, act):
        """ResNetBasicHead (head_helper.py:198-223): global pooling when the AvgPool3d kernel covers the feature map
        (or is adaptive), else fully-convolutional inference over the remaining positions."""
        sizes = self.head.pool_size
        full = all(ps is None or [int(v) for v in ps] == list(x.shape[1:4]) for x, ps in zip(xs, sizes))
        if full:
            return plan.head(xs, self.head.projection.weight, self.head.projection.bias, act)
        for x, ps in zip(xs, sizes):
            if ps is None or any(int(k) > n for k, n in zip(ps, x.shape[1:4])):
                raise NotImplementedError("head AvgPool3d kernel %s does not fit the feature map %s"
                                          % (ps, list(x.shape[1:4])))
        return plan.head_positions(xs, sizes, self.head.projection.weight, self.head.projection.bias, act)

    def _emit_roi_head(self, plan, xs, act):
        """ResNetRoIHead.forward (head_helper.py:100-130) in two parts.  In the plan (CUDA graph): the temporal
        AvgPool3d of every pathway's res5 output into an FP32 map.  Per call, outside the graph (Plan.run_boxes):
        RoIAlign + spatial max of every pathway into one FP32 row per box, then Linear + activation."""
        maps, scales, res = [], [], []
        for p, x in enumerate(xs):
            roi = getattr(self.head, "s%d_roi" % p)
            r = [int(v) for v in roi.output_size]
            if r[0] != r[1] or roi.sampling_ratio != 0:
                raise NotImplementedError("ROIAlign output %s / sampling_ratio %d: the kernel covers square outputs "
                                          "with the adaptive grid (sampling_ratio 0) of ResNetRoIHead" % (r, roi.sampling_ratio))
            maps.append(plan.temporal_mean(x))
            scales.append(roi.spatial_scale)
            res.append(r[0])
        plan.roi_head(maps, scales, res, bool(self.head.s0_roi.aligned), self.head.projection.weight,
                      self.head.projection.bias, act)

    def _emit_stage_pathway(self, plan, stage, pw, x, dst, stride, dil):
        """One pathway of ResStage.forward (resnet_helper.py:530-561): residual blocks, each optionally followed by
        its Nonlocal block; the units ping-pong between two scratch activations and the last one writes `dst`."""
        units = []
        for bi in range(stage.num_blocks[pw]):
            units.append(("res", getattr(stage, "pathway{}_res{}".format(pw, bi)), stride if bi == 0 else 1))
            nln = getattr(stage, "pathway{}_nonlocal{}".format(pw, bi), None)
            if nln is not None:
                units.append(("nonlocal", nln, None))
        B, T, Ho, Wo, co = dst.shape
        ping = [plan.act(B, T, Ho, Wo, co) for _ in range(min(2, len(units) - 1))]
        for ui, (kind, mod, st) in enumerate(units):
            y = dst if ui == len(units) - 1 else ping[ui % 2]
            if kind == "res":
                self._emit_block(plan, mod, x, y, st, dil)
            else:
                plan.nonlocal_block(x, y, mod, group=stage.nonlocal_group[pw])
            x = y

    def _emit_block(self, plan, blk, x, y, stride, dil):
        """ResBlock (resnet_helper.py:352-358): y = relu(shortcut(x) + bn(c(relu(bn(b(relu(bn(a(x))))))))).
        4 (or 3) implicit-GEMM launches; BN folded, ReLU and the residual add in the epilogues."""
        t = blk.branch2
        B, T, H, W, _ = x.shape
        _, _, Ho, Wo, co = y.shape
        ci = t.a.out_channels
        s1 = t.a.stride[1]
        Ha, Wa = (H - 1) // s1 + 1, (W - 1) // s1 + 1   # Tx1x1 conv, stride (1,s1,s1), no spatial padding
        ta = plan.act(B, T, Ha, Wa, ci, role="operand")      # read by the next convolution only
        tb = plan.act(B, T, Ho, Wo, ci, role="operand")
        if hasattr(blk, "branch1"):
            sc = plan.act(B, T, Ho, Wo, co, role="residual")  # read by conv c's residual add only
            w, b = plan.once(fold_conv_bn, blk.branch1.weight, None, blk.branch1_bn)
            plan.conv(x, sc, w, b, stride=tuple(blk.branch1.stride))
        else:
            sc = x
        w, b = plan.once(fold_conv_bn, t.a.weight, None, t.a_bn)
        plan.conv(x, ta, w, b, stride=tuple(t.a.stride), padding=tuple(t.a.padding), act=rt.ACT_RELU)
        # RESNET.NUM_GROUPS > 1 (ResNeXt, resnet_helper.py:196-205): Plan.conv runs one implicit GEMM per group on
        # channel slices, or one dense GEMM over a block-diagonal weight when the slices are thinner than a TMA row;
        # PrecisePlan.conv always takes the block-diagonal weight
        w, b = plan.once(fold_conv_bn, t.b.weight, None, t.b_bn)
        plan.conv(ta, tb, w, b, stride=tuple(t.b.stride), padding=tuple(t.b.padding),
                  dilation=tuple(t.b.dilation), groups=t.b.groups, act=rt.ACT_RELU)
        w, b = plan.once(fold_conv_bn, t.c.weight, None, t.c_bn)
        plan.conv(tb, y, w, b, act=rt.ACT_RELU, res=sc)

@MODEL_REGISTRY.register()
class SlowFastDualAttention(_TwoStreamResNet):
    """custom_video_model_builder.py:171-445."""

    def __init__(self, cfg):
        super().__init__()
        self._build(cfg, dual_attention=True)


@MODEL_REGISTRY.register()
class SlowFast(_TwoStreamResNet):
    """video_model_builder.py:153-416."""

    def __init__(self, cfg):
        super().__init__()
        self._build(cfg, dual_attention=False)


@MODEL_REGISTRY.register()
class ResNet(_TwoStreamResNet):
    """video_model_builder.py:419-611: single-pathway ResNet (C2D, I3D, Slow) without lateral connections.  Same
    stem / bottleneck / head kernels as the two-stream models; the max-pool after res2 is real here (kernel = stride =
    _POOL1[arch], e.g. (2,1,1) for c2d / i3d).  Nonlocal blocks (C2D_NLN / I3D_NLN / SLOW_NLN): engine.nonlocal_block."""

    num_pathways = 1

    def __init__(self, cfg):
        super().__init__()
        assert cfg.MODEL.ARCH in _POOL1.keys()
        pool_size = _POOL1[cfg.MODEL.ARCH]
        assert len({len(pool_size), self.num_pathways}) == 1
        assert cfg.RESNET.DEPTH in _MODEL_STAGE_DEPTH.keys()
        self.norm_module = get_norm(cfg)
        self.enable_detection = bool(cfg.DETECTION.ENABLE)
        depths = _MODEL_STAGE_DEPTH[cfg.RESNET.DEPTH]
        num_groups, wpg = cfg.RESNET.NUM_GROUPS, cfg.RESNET.WIDTH_PER_GROUP
        dim_inner = num_groups * wpg
        tk = _TEMPORAL_KERNEL_BASIS[cfg.MODEL.ARCH]
        self.s1 = VideoModelStem(dim_in=cfg.DATA.INPUT_CHANNEL_NUM, dim_out=[wpg], kernel=[tk[0][0] + [7, 7]],
                                 stride=[[1, 2, 2]], padding=[[tk[0][0][0] // 2, 3, 3]], norm_module=self.norm_module)
        c_prev = wpg
        for i, name in enumerate(("s2", "s3", "s4", "s5")):
            c_out = wpg * 4 * (2 ** i)
            setattr(self, name, ResStage(
                dim_in=[c_prev], dim_out=[c_out], dim_inner=[dim_inner * (2 ** i)], temp_kernel_sizes=tk[i + 1],
                stride=cfg.RESNET.SPATIAL_STRIDES[i], num_blocks=[depths[i]], num_groups=[num_groups],
                num_block_temp_kernel=cfg.RESNET.NUM_BLOCK_TEMP_KERNEL[i], nonlocal_inds=cfg.NONLOCAL.LOCATION[i], nonlocal_group=cfg.NONLOCAL.GROUP[i],
                nonlocal_pool=cfg.NONLOCAL.POOL[i], instantiation=cfg.NONLOCAL.INSTANTIATION,
                dilation=cfg.RESNET.SPATIAL_DILATIONS[i], trans_func_name=cfg.RESNET.TRANS_FUNC,
                stride_1x1=cfg.RESNET.STRIDE_1X1, norm_module=self.norm_module))
            if name == "s2":
                self.add_module("pathway0_pool",
                                nn.MaxPool3d(kernel_size=pool_size[0], stride=pool_size[0], padding=[0, 0, 0]))
            c_prev = c_out
        if self.enable_detection:      # video_model_builder.py: ResNetRoIHead branch of ResNet._construct_network
            R = cfg.DETECTION.ROI_XFORM_RESOLUTION
            self.head = ResNetRoIHead(
                dim_in=[wpg * 32], num_classes=cfg.MODEL.NUM_CLASSES,
                pool_size=[[cfg.DATA.NUM_FRAMES // pool_size[0][0], 1, 1]], resolution=[[R] * 2],
                scale_factor=[cfg.DETECTION.SPATIAL_SCALE_FACTOR], dropout_rate=cfg.MODEL.DROPOUT_RATE,
                act_func=cfg.MODEL.HEAD_ACT, aligned=cfg.DETECTION.ALIGNED)
        else:
            if cfg.MULTIGRID.SHORT_CYCLE:
                head_pool = [None, None]    # as in the reference (video_model_builder.py:584-586): the head then rejects it
            else:
                c = cfg.DATA.CROP_SIZE // 32
                head_pool = [[cfg.DATA.NUM_FRAMES // pool_size[0][0], c // pool_size[0][1], c // pool_size[0][2]]]
            self.head = ResNetBasicHead(dim_in=[wpg * 32], num_classes=cfg.MODEL.NUM_CLASSES, pool_size=head_pool,
                                        dropout_rate=cfg.MODEL.DROPOUT_RATE, act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    def _compile(self, plan):
        cfg = self._cfg
        x = plan.inputs[0]
        B, _, T, H, W = x.shape
        wpg = cfg.RESNET.WIDTH_PER_GROUP

        def conv_out(n, k, s, p, d=1):
            return (n + 2 * p - d * (k - 1) - 1) // s + 1

        stem = self.s1.pathway0_stem
        k, s, p = stem.kernel, stem.stride, stem.padding
        To, Ho, Wo = conv_out(T, k[0], s[0], p[0]), conv_out(H, k[1], s[1], p[1]), conv_out(W, k[2], s[2], p[2])
        y = plan.act(B, To, Ho, Wo, wpg)
        w, b = plan.once(fold_conv_bn, stem.conv.weight, None, stem.bn)
        plan.stem(x, y, w, b, tuple(s), tuple(p), act=rt.ACT_RELU)
        cur = plan.act(B, To, conv_out(Ho, 3, 2, 1), conv_out(Wo, 3, 2, 1), wpg, name="s1_cat0")
        plan.pool(y, cur, (1, 3, 3), (1, 2, 2), (0, 1, 1))
        for i, name in enumerate(("s2", "s3", "s4", "s5")):
            stage = getattr(self, name)
            co = wpg * 4 * (2 ** i)
            stride, dil = cfg.RESNET.SPATIAL_STRIDES[i][0], cfg.RESNET.SPATIAL_DILATIONS[i][0]
            _, T, H, W, _ = cur.shape
            Ho, Wo = conv_out(H, 1, stride, 0), conv_out(W, 1, stride, 0)
            dst = plan.act(B, T, Ho, Wo, co, name="%s_cat0" % name)
            self._emit_stage_pathway(plan, stage, 0, cur, dst, stride, dil)
            cur = dst
            if name == "s2":
                ks = [int(v) for v in self.pathway0_pool.kernel_size]
                if ks != [1, 1, 1]:
                    _, T, H, W, _ = cur.shape
                    pooled = plan.act(B, (T - ks[0]) // ks[0] + 1, (H - ks[1]) // ks[1] + 1, (W - ks[2]) // ks[2] + 1, co,
                                      name="s2_pool0")
                    plan.pool(cur, pooled, tuple(ks), tuple(ks), (0, 0, 0))
                    cur = pooled
        act = {"softmax": rt.HEAD_SOFTMAX, "sigmoid": rt.HEAD_SIGMOID}[self.head.act_func]
        if self.enable_detection:
            return self._emit_roi_head(plan, [cur], act)
        self._emit_head(plan, [cur], act)
