"""The efficient two-stream models of the reference behind the same registry / nn.Module surface:

  SlowFastShuffleNetV2   (SlowFast/slowfast/models/custom_video_model_builder.py:448-617)
  SlowFastShuffleNet     (custom_video_model_builder.py:620-789)

Same contract as nets_resnet.py: the module tree only holds parameters under the reference's state_dict keys
(SURVEY.md Appendix D: `s#.pathway#_channel_<C>.features.#.banch{1,2}.#.*`, `...conv{1,2,3}.weight`, ...); the
arithmetic is a launch plan of libesf_b200 kernels.  These backbones have channel counts that are not multiples of 8
(27, 54, 6, ...), so most of their layers run on the CUDA-core kernels (`esf_conv_direct`, `esf_pool3d`,
`esf_shuffle_concat`); layers whose views happen to be 16-byte addressable go to the tensor-core implicit GEMM
automatically (engine.Plan.conv).
"""
import math

import torch
import torch.nn as nn

from . import runtime as rt
from .build import MODEL_REGISTRY
from .engine import fold_conv_bn
from .nets_resnet import FuseFastAndSlow, _Holder, _PlannedModel, get_norm, init_weights


def _stage_init(module):
    """The per-stage `_initialize_weights` of the reference helpers (e.g. shufflenetv2_helper.py:283-297): conv weights
    ~ N(0, 2 / (k_t k_h k_w C_out)), BN weight 1 / bias 0, Linear N(0, 0.01).  Run at the same points of construction
    as in the reference so that a given torch seed produces the same weights."""
    for m in module.modules():
        if isinstance(m, nn.Conv3d):
            n = m.kernel_size[0] * m.kernel_size[1] * m.kernel_size[2] * m.out_channels
            m.weight.data.normal_(0, math.sqrt(2.0 / n))
            if m.bias is not None:
                m.bias.data.zero_()
        elif isinstance(m, nn.BatchNorm3d):
            m.weight.data.fill_(1)
            m.bias.data.zero_()
        elif isinstance(m, nn.Linear):
            m.weight.data.normal_(0, 0.01)
            m.bias.data.zero_()


def _conv_out(n, k, s, p, d=1):
    return (n + 2 * p - d * (k - 1) - 1) // s + 1


class _EfficientBase(_PlannedModel):
    """Plan-emission helpers shared by the efficient models."""

    def _emit_conv(self, plan, x, conv, bn, act, y=None, res=None, name=None):
        """conv (+BN) (+act) of one nn.Conv3d; allocates the output when `y` is None."""
        B, T, H, W, _ = x.shape
        k, s, p, d = conv.kernel_size, conv.stride, conv.padding, conv.dilation
        To, Ho, Wo = (_conv_out(T, k[0], s[0], p[0], d[0]), _conv_out(H, k[1], s[1], p[1], d[1]),
                      _conv_out(W, k[2], s[2], p[2], d[2]))
        if y is None:
            y = plan.act(B, To, Ho, Wo, conv.out_channels, name=name)
        w, b = plan.once(fold_conv_bn, conv.weight, conv.bias, bn)
        plan.conv(x, y, w, b, stride=tuple(s), padding=tuple(p), dilation=tuple(d), groups=conv.groups, act=act, res=res)
        return y

    def _emit_stem(self, plan, seq, x_nc, dst, act):
        """Sequential(Conv3d, BN, ReLU|ReLU6[, MaxPool3d]) on the FP32 clip; writes into `dst` (a concat slice)."""
        conv, bn = seq[0], seq[1]
        B, _, T, H, W = x_nc.shape
        k, s, p = conv.kernel_size, conv.stride, conv.padding
        To, Ho, Wo = _conv_out(T, k[0], s[0], p[0]), _conv_out(H, k[1], s[1], p[1]), _conv_out(W, k[2], s[2], p[2])
        w, b = plan.once(fold_conv_bn, conv.weight, conv.bias, bn)
        pool = seq[3] if len(seq) > 3 else None
        if pool is None:
            y = plan.act(B, To, Ho, Wo, conv.out_channels)
            plan.stem(x_nc, y, w, b, tuple(s), tuple(p), act=act)
            plan.shuffle_concat(y, None, 1, dst)   # plain copy into the slice (groups = 1)
            return
        y = plan.act(B, To, Ho, Wo, conv.out_channels)
        plan.stem(x_nc, y, w, b, tuple(s), tuple(p), act=act)
        pk = pool.kernel_size if isinstance(pool.kernel_size, (tuple, list)) else (pool.kernel_size,) * 3
        ps = pool.stride if isinstance(pool.stride, (tuple, list)) else (pool.stride,) * 3
        pp = pool.padding if isinstance(pool.padding, (tuple, list)) else (pool.padding,) * 3
        plan.pool(y, dst, tuple(pk), tuple(ps), tuple(pp))

    @staticmethod
    def _pooled_shape(T, H, W, seq):
        conv = seq[0]
        k, s, p = conv.kernel_size, conv.stride, conv.padding
        T, H, W = _conv_out(T, k[0], s[0], p[0]), _conv_out(H, k[1], s[1], p[1]), _conv_out(W, k[2], s[2], p[2])
        if len(seq) > 3:
            pool = seq[3]
            pk = pool.kernel_size if isinstance(pool.kernel_size, (tuple, list)) else (pool.kernel_size,) * 3
            ps = pool.stride if isinstance(pool.stride, (tuple, list)) else (pool.stride,) * 3
            pp = pool.padding if isinstance(pool.padding, (tuple, list)) else (pool.padding,) * 3
            T, H, W = _conv_out(T, pk[0], ps[0], pp[0]), _conv_out(H, pk[1], ps[1], pp[1]), _conv_out(W, pk[2], ps[2], pp[2])
        return T, H, W


# ================================================================================================ ShuffleNetV2
class InvertedResidual(_Holder):
    """shufflenetv2_helper.py:46-112 (sic: 'banch')."""

    def __init__(self, inp, oup, stride):
        super().__init__()
        self.stride = stride
        assert stride in [1, 2]
        oup_inc = oup // 2
        if self.stride == 1:
            self.banch2 = nn.Sequential(
                nn.Conv3d(oup_inc, oup_inc, 1, 1, 0, bias=False), nn.BatchNorm3d(oup_inc), nn.ReLU(inplace=True),
                nn.Conv3d(oup_inc, oup_inc, 3, (1, stride, stride), 1, groups=oup_inc, bias=False),
                nn.BatchNorm3d(oup_inc),
                nn.Conv3d(oup_inc, oup_inc, 1, 1, 0, bias=False), nn.BatchNorm3d(oup_inc), nn.ReLU(inplace=True))
        else:
            self.banch1 = nn.Sequential(
                nn.Conv3d(inp, inp, 3, (1, stride, stride), 1, groups=inp, bias=False), nn.BatchNorm3d(inp),
                nn.Conv3d(inp, oup_inc, 1, 1, 0, bias=False), nn.BatchNorm3d(oup_inc), nn.ReLU(inplace=True))
            self.banch2 = nn.Sequential(
                nn.Conv3d(inp, oup_inc, 1, 1, 0, bias=False), nn.BatchNorm3d(oup_inc), nn.ReLU(inplace=True),
                nn.Conv3d(oup_inc, oup_inc, 3, (1, stride, stride), 1, groups=oup_inc, bias=False),
                nn.BatchNorm3d(oup_inc),
                nn.Conv3d(oup_inc, oup_inc, 1, 1, 0, bias=False), nn.BatchNorm3d(oup_inc), nn.ReLU(inplace=True))


class ShuffleNetV2_Inverted_Residual_Block(_Holder):
    """shufflenetv2_helper.py:178-219."""

    def __init__(self, input_channel, idxstage, stage_out_channels):
        super().__init__()
        self.stage_repeats = [4, 8, 4]
        feats = []
        output_channel = stage_out_channels[idxstage + 2]
        for i in range(self.stage_repeats[idxstage]):
            feats.append(InvertedResidual(input_channel, output_channel, 2 if i == 0 else 1))
            input_channel = output_channel
        self.features = nn.Sequential(*feats)
        _stage_init(self)


class ShuffleNetV2_Stage(_Holder):
    """shufflenetv2_helper.py:222-297."""

    def __init__(self, input_channel, idxstage, slow_stage_out_channels, fast_stage_out_channels):
        super().__init__()
        self.idxstage = idxstage
        self.num_pathways = len(input_channel)
        self.out_channels = [slow_stage_out_channels[idxstage + 2], fast_stage_out_channels[idxstage + 2]]
        for p, chans in enumerate((slow_stage_out_channels, fast_stage_out_channels)):
            blk = ShuffleNetV2_Inverted_Residual_Block(input_channel[p], idxstage, chans)
            self.add_module("pathway{}_channel_{}".format(p, chans[idxstage + 2]), blk)
            _stage_init(self)

    def pathway(self, p):
        return getattr(self, "pathway{}_channel_{}".format(p, self.out_channels[p]))


class ShuffleNetV2_Model_Stem(_Holder):
    """stem_helper.py:237-270: Conv3d 3x3x3 s(1,2,2) p1 -> BN -> ReLU -> MaxPool3d k3 s(1,2,2) p1."""

    def __init__(self, input_channels, img_dim=3):
        super().__init__()
        self.num_pathways = len(input_channels)
        for p in range(self.num_pathways):
            stem = nn.Sequential(
                nn.Conv3d(img_dim, input_channels[p], kernel_size=3, stride=(1, 2, 2), padding=(1, 1, 1), bias=False),
                nn.BatchNorm3d(input_channels[p]), nn.ReLU(inplace=True),
                nn.MaxPool3d(kernel_size=3, stride=(1, 2, 2), padding=1))
            self.add_module("pathway{}_stem".format(p), stem)


class ShuffleNetV2BasicHead(_Holder):
    """head_helper.py:499-557: per pathway 1x1x1 conv + BN + ReLU -> global avg pool -> cat -> Dropout -> Linear ->
    softmax -> mean."""

    def __init__(self, input_channel, last_channel, num_classes, dropout_rate, act_func="softmax"):
        super().__init__()
        self.num_pathways = len(input_channel)
        for p in range(self.num_pathways):
            feats = nn.Sequential(nn.Sequential(
                nn.Conv3d(input_channel[p], last_channel[p], 1, 1, 0, bias=False), nn.BatchNorm3d(last_channel[p]),
                nn.ReLU(inplace=True)))
            self.add_module("pathway{}_conv1x1x1".format(p), feats)
        if act_func == "softmax":
            self.act = nn.Softmax(dim=4)
        elif act_func == "sigmoid":
            self.act = nn.Sigmoid()
        self.act_func = act_func
        self.classifier = nn.Sequential(nn.Dropout(dropout_rate), nn.Linear(sum(last_channel), num_classes, bias=True))


@MODEL_REGISTRY.register()
class SlowFastShuffleNetV2(_EfficientBase):
    """custom_video_model_builder.py:448-617."""

    def __init__(self, cfg):
        super().__init__()
        self.norm_module = get_norm(cfg)
        if cfg.DETECTION.ENABLE:
            raise NotImplementedError("DETECTION.ENABLE is out of scope")
        self.enable_detection = False
        width_mult = cfg.SLOWFAST.WIDTH_MULTI
        table = {0.25: [-1, 24, 32, 64, 128, 1024], 0.5: [-1, 24, 48, 96, 192, 1024],
                 1.0: [-1, 24, 116, 240, 464, 1024],   # 232 -> 240 in the reference (:476)
                 1.5: [-1, 24, 176, 352, 704, 1024], 2.0: [-1, 24, 224, 496, 976, 2048]}  # 488 -> 496 (:480)
        if width_mult not in table:
            raise ValueError("{} groups is not supported for 1x1 Grouped Convolutions".format(width_mult))
        self.stage_out_channels = table[width_mult]
        beta = cfg.SLOWFAST.BETA_INV
        self.fast_stage_out_channels = [c // beta for c in self.stage_out_channels]
        so, fo = self.stage_out_channels, self.fast_stage_out_channels
        self.s1 = ShuffleNetV2_Model_Stem(input_channels=[so[1], so[1] // beta], img_dim=len(cfg.DATA.MEAN))
        for i in range(1, 5):
            fuse = FuseFastAndSlow(dim_in=[so[i], fo[i]], alpha=cfg.SLOWFAST.ALPHA, beta_inv=beta,
                                   norm_module=self.norm_module)
            setattr(self, "s%d_fuse" % i, fuse)
            if i < 4:
                stage = ShuffleNetV2_Stage(input_channel=[so[i] + fo[i], fo[i] + so[i] // beta], idxstage=i - 1,
                                           slow_stage_out_channels=so, fast_stage_out_channels=fo)
                setattr(self, "s%d" % (i + 1), stage)
        self.head = ShuffleNetV2BasicHead(
            input_channel=[so[4] + fo[4], fo[4] + so[4] // beta], last_channel=[so[-1], fo[-1]],
            num_classes=cfg.MODEL.NUM_CLASSES, dropout_rate=cfg.MODEL.DROPOUT_RATE, act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    # child order of the reference: s1, s1_fuse, s2, s2_fuse, s3, s3_fuse, s4, s4_fuse, head -- setattr order above
    # registers s1_fuse before s2 etc., matching it.

    def _emit_unit(self, plan, unit, x, y):
        """InvertedResidual.forward (shufflenetv2_helper.py:104-112)."""
        if unit.stride == 1:
            c = x.shape[4] // 2
            x1, x2 = x[..., :c], x[..., c:]
            b2 = unit.banch2
            t = self._emit_conv(plan, x2, b2[0], b2[1], rt.ACT_RELU)
            t = self._emit_conv(plan, t, b2[3], b2[4], rt.ACT_NONE)
            t = self._emit_conv(plan, t, b2[5], b2[6], rt.ACT_RELU)
            plan.shuffle_concat(x1, t, 2, y)
        else:
            b1, b2 = unit.banch1, unit.banch2
            u = self._emit_conv(plan, x, b1[0], b1[1], rt.ACT_NONE)
            u = self._emit_conv(plan, u, b1[2], b1[3], rt.ACT_RELU)
            t = self._emit_conv(plan, x, b2[0], b2[1], rt.ACT_RELU)
            t = self._emit_conv(plan, t, b2[3], b2[4], rt.ACT_NONE)
            t = self._emit_conv(plan, t, b2[5], b2[6], rt.ACT_RELU)
            plan.shuffle_concat(u, t, 2, y)

    def _compile(self, plan):
        cfg = self._cfg
        alpha, beta = cfg.SLOWFAST.ALPHA, cfg.SLOWFAST.BETA_INV
        so, fo = self.stage_out_channels, self.fast_stage_out_channels
        xs_in = plan.inputs
        B = xs_in[0].shape[0]
        assert xs_in[1].shape[2] == xs_in[0].shape[2] * alpha, "fast pathway must have ALPHA x the frames of the slow one"
        # concat buffers after stage i: slow [x_s (so) | from_fast (fo)], fast [from_slow (so // beta) | x_f (fo)]
        cur = []
        for p in range(2):
            seq = getattr(self.s1, "pathway{}_stem".format(p))
            _, _, T, H, W = xs_in[p].shape
            T, H, W = self._pooled_shape(T, H, W, seq)
            c_own = so[1] if p == 0 else fo[1]
            tot = so[1] + fo[1] if p == 0 else so[1] // beta + fo[1]
            off = 0 if p == 0 else so[1] // beta
            buf = plan.act(B, T, H, W, tot, name="s1_cat%d" % p)
            self._emit_stem(plan, seq, xs_in[p], buf[..., off:off + c_own], rt.ACT_RELU)
            cur.append((buf, off, c_own))
        self._emit_fuse(plan, self.s1_fuse, cur)
        for i in range(1, 4):
            stage = getattr(self, "s%d" % (i + 1))
            nxt = []
            for p in range(2):
                x = cur[p][0]
                c_own = so[i + 1] if p == 0 else fo[i + 1]
                tot = so[i + 1] + fo[i + 1] if p == 0 else so[i + 1] // beta + fo[i + 1]
                off = 0 if p == 0 else so[i + 1] // beta
                units = stage.pathway(p).features
                _, T, H, W, _ = x.shape
                Ho, Wo = _conv_out(H, 3, 2, 1), _conv_out(W, 3, 2, 1)
                dst = plan.act(B, T, Ho, Wo, tot, name="s%d_cat%d" % (i + 1, p))
                for ui, unit in enumerate(units):
                    last = ui == len(units) - 1
                    y = dst[..., off:off + c_own] if last else plan.act(B, T, Ho, Wo, c_own)
                    self._emit_unit(plan, unit, x, y)
                    x = y
                nxt.append((dst, off, c_own))
            cur = nxt
            self._emit_fuse(plan, getattr(self, "s%d_fuse" % (i + 1)), cur)
        feats = []
        for p in range(2):
            seq = getattr(self.head, "pathway{}_conv1x1x1".format(p))[0]
            feats.append(self._emit_conv(plan, cur[p][0], seq[0], seq[1], rt.ACT_RELU))
        act = {"softmax": rt.HEAD_SOFTMAX, "sigmoid": rt.HEAD_SIGMOID}[self.head.act_func]
        lin = self.head.classifier[1]
        plan.head(feats, lin.weight, lin.bias, act)


# ================================================================================================ ShuffleNet (v1)
class Bottleneck(_Holder):
    """shufflenet_helper.py:37-84."""

    def __init__(self, in_planes, out_planes, stride, groups):
        super().__init__()
        self.stride = stride
        self.groups = groups
        mid_planes = out_planes // 4
        if self.stride == 2:
            mid_planes = out_planes // 2
            out_planes = out_planes - out_planes // 2
        g = 1 if in_planes == 24 else groups
        self.conv1 = nn.Conv3d(in_planes, mid_planes, kernel_size=1, groups=g, bias=False)
        self.bn1 = nn.BatchNorm3d(mid_planes)
        self.conv2 = nn.Conv3d(mid_planes, mid_planes, kernel_size=(3, 3, 3), stride=(1, stride, stride), padding=1,
                               groups=mid_planes, bias=False)
        self.bn2 = nn.BatchNorm3d(mid_planes)
        self.conv3 = nn.Conv3d(mid_planes, out_planes, kernel_size=1, groups=groups, bias=False)
        self.bn3 = nn.BatchNorm3d(out_planes)
        self.relu = nn.ReLU(inplace=True)
        if stride == 2:
            self.shortcut = nn.Sequential(
                nn.Conv3d(in_planes, mid_planes, kernel_size=1, bias=False),
                nn.AvgPool3d(kernel_size=(1, 3, 3), stride=(1, 2, 2), padding=(0, 1, 1)))


class ShuffleNet_Residual_Block(_Holder):
    """shufflenet_helper.py:165-218."""

    def __init__(self, in_plane, out_plane, num_block, group):
        super().__init__()
        layers = []
        for i in range(num_block):
            layers.append(Bottleneck(in_plane, out_plane, stride=2 if i == 0 else 1, groups=group))
            in_plane = out_plane
        self.features = nn.Sequential(*layers)
        _stage_init(self)


class ShuffleNet_Stage(_Holder):
    """shufflenet_helper.py:221-295."""

    def __init__(self, input_channel, slow_stage_out_channels, fast_stage_out_channels, num_block, group):
        super().__init__()
        self.out_channels = [slow_stage_out_channels, fast_stage_out_channels]
        self.num_pathways = len(input_channel)
        for p in range(self.num_pathways):
            blk = ShuffleNet_Residual_Block(input_channel[p], self.out_channels[p], num_block, group)
            self.add_module("pathway{}_channel_{}".format(p, self.out_channels[p]), blk)
            _stage_init(self)

    def pathway(self, p):
        return getattr(self, "pathway{}_channel_{}".format(p, self.out_channels[p]))


class ShuffleNet_Model_Stem(ShuffleNetV2_Model_Stem):
    """stem_helper.py:274-306 (same layers as the ShuffleNetV2 stem)."""


class ShuffleNetBasicHead(_Holder):
    """head_helper.py:562-609: global avg pool per pathway -> cat -> Dropout -> Linear -> softmax -> mean."""

    def __init__(self, input_channel, num_classes, dropout_rate, act_func="softmax"):
        super().__init__()
        self.num_pathways = len(input_channel)
        if act_func == "softmax":
            self.act = nn.Softmax(dim=4)
        elif act_func == "sigmoid":
            self.act = nn.Sigmoid()
        self.act_func = act_func
        self.classifier = nn.Sequential(nn.Dropout(dropout_rate), nn.Linear(sum(input_channel), num_classes, bias=True))


@MODEL_REGISTRY.register()
class SlowFastShuffleNet(_EfficientBase):
    """custom_video_model_builder.py:620-789."""

    def __init__(self, cfg):
        super().__init__()
        self.norm_module = get_norm(cfg)
        if cfg.DETECTION.ENABLE:
            raise NotImplementedError("DETECTION.ENABLE is out of scope")
        self.enable_detection = False
        groups = cfg.SLOWFAST.GROUPS
        self.num_blocks = [4, 8, 4]
        self.groups = groups
        table = {1: [24, 144, 288, 567], 2: [24, 200, 400, 800], 3: [24, 240, 480, 960], 4: [24, 272, 544, 1088],
                 8: [24, 384, 768, 1536]}
        if groups not in table:
            raise ValueError("{} groups is not supported for 1x1 Grouped Convolutions".format(groups))
        beta = cfg.SLOWFAST.BETA_INV
        self.stage_out_channels = [int(i * cfg.SLOWFAST.WIDTH_MULTI) for i in table[groups]]
        self.fast_stage_out_channels = [c // beta for c in self.stage_out_channels]
        so, fo = self.stage_out_channels, self.fast_stage_out_channels
        self.s1 = ShuffleNet_Model_Stem(input_channels=[so[0], fo[0]], img_dim=len(cfg.DATA.MEAN))
        for i in range(4):
            fuse = FuseFastAndSlow(dim_in=[so[i], fo[i]], alpha=cfg.SLOWFAST.ALPHA, beta_inv=beta,
                                   norm_module=self.norm_module)
            setattr(self, "s%d_fuse" % (i + 1), fuse)
            if i < 3:
                stage = ShuffleNet_Stage(input_channel=[so[i] + fo[i], fo[i] + so[i] // beta],
                                         slow_stage_out_channels=so[i + 1], fast_stage_out_channels=fo[i + 1],
                                         num_block=self.num_blocks[i], group=groups)
                setattr(self, "s%d" % (i + 2), stage)
        self.head = ShuffleNetBasicHead(input_channel=[so[3] + fo[3], fo[3] + so[3] // beta],
                                        num_classes=cfg.MODEL.NUM_CLASSES, dropout_rate=cfg.MODEL.DROPOUT_RATE,
                                        act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    def _emit_unit(self, plan, blk, x, y):
        """Bottleneck.forward (shufflenet_helper.py:75-84)."""
        conv1 = blk.conv1
        if (blk.groups > 1 and tuple(conv1.kernel_size) == (1, 1, 1) and x.shape[4] >= 8
                and conv1.out_channels % blk.groups == 0):
            # channel_shuffle(relu(bn(conv1(x)))) is a permutation of conv1's output channels: fold it into the ORDER of
            # the weight rows.  A permuted grouped conv is no longer grouped, so the layer runs as one dense implicit
            # GEMM over a block-diagonal weight (the layers are HBM bound; `groups`-fold MACs on structural zeros) --
            # one launch instead of a GEMM per group plus the shuffle kernel (1.6 ms of the 12.3 ms ShuffleNet step).
            w, b = plan.once(fold_conv_bn, conv1.weight, conv1.bias, blk.bn1)
            cout, cin_g, g = w.shape[0], w.shape[1], conv1.groups
            wd = torch.zeros((cout, cin_g * g, 1, 1, 1), dtype=w.dtype, device=w.device)
            for i in range(g):
                rows = slice(i * (cout // g), (i + 1) * (cout // g))
                wd[rows, i * cin_g:(i + 1) * cin_g] = w[rows]
            G, cpg = blk.groups, cout // blk.groups
            src = torch.tensor([(o % G) * cpg + o // G for o in range(cout)], device=w.device)   # shuffled[o] = y[src[o]]
            t = plan.act(*x.shape[:4], cout)
            plan.conv(x, t, wd[src], b[src], act=rt.ACT_RELU)
        else:
            t = self._emit_conv(plan, x, conv1, blk.bn1, rt.ACT_RELU)
            if blk.groups > 1:
                ts = plan.act(*t.shape)
                plan.shuffle_concat(t, None, blk.groups, ts)
                t = ts
        t = self._emit_conv(plan, t, blk.conv2, blk.bn2, rt.ACT_NONE)
        if blk.stride == 2:
            c3 = blk.conv3.out_channels
            self._emit_conv(plan, t, blk.conv3, blk.bn3, rt.ACT_RELU, y=y[..., :c3])      # relu(cat) == cat(relu)
            sc = self._emit_conv(plan, x, blk.shortcut[0], None, rt.ACT_NONE)
            plan.pool(sc, y[..., c3:], (1, 3, 3), (1, 2, 2), (0, 1, 1), is_avg=True, act=rt.ACT_RELU)
        else:
            self._emit_conv(plan, t, blk.conv3, blk.bn3, rt.ACT_RELU, y=y, res=x)

    def _compile(self, plan):
        cfg = self._cfg
        alpha, beta = cfg.SLOWFAST.ALPHA, cfg.SLOWFAST.BETA_INV
        so, fo = self.stage_out_channels, self.fast_stage_out_channels
        xs_in = plan.inputs
        B = xs_in[0].shape[0]
        assert xs_in[1].shape[2] == xs_in[0].shape[2] * alpha, "fast pathway must have ALPHA x the frames of the slow one"
        cur = []
        for p in range(2):
            seq = getattr(self.s1, "pathway{}_stem".format(p))
            _, _, T, H, W = xs_in[p].shape
            T, H, W = self._pooled_shape(T, H, W, seq)
            c_own = so[0] if p == 0 else fo[0]
            tot = so[0] + fo[0] if p == 0 else so[0] // beta + fo[0]
            off = 0 if p == 0 else so[0] // beta
            buf = plan.act(B, T, H, W, tot, name="s1_cat%d" % p)
            self._emit_stem(plan, seq, xs_in[p], buf[..., off:off + c_own], rt.ACT_RELU)
            cur.append((buf, off, c_own))
        self._emit_fuse(plan, self.s1_fuse, cur)
        for i in range(3):
            stage = getattr(self, "s%d" % (i + 2))
            nxt = []
            for p in range(2):
                x = cur[p][0]
                c_own = so[i + 1] if p == 0 else fo[i + 1]
                tot = so[i + 1] + fo[i + 1] if p == 0 else so[i + 1] // beta + fo[i + 1]
                off = 0 if p == 0 else so[i + 1] // beta
                units = stage.pathway(p).features
                _, T, H, W, _ = x.shape
                Ho, Wo = _conv_out(H, 3, 2, 1), _conv_out(W, 3, 2, 1)
                dst = plan.act(B, T, Ho, Wo, tot, name="s%d_cat%d" % (i + 2, p))
                for ui, unit in enumerate(units):
                    last = ui == len(units) - 1
                    y = dst[..., off:off + c_own] if last else plan.act(B, T, Ho, Wo, c_own)
                    self._emit_unit(plan, unit, x, y)
                    x = y
                nxt.append((dst, off, c_own))
            cur = nxt
            self._emit_fuse(plan, getattr(self, "s%d_fuse" % (i + 2)), cur)
        act = {"softmax": rt.HEAD_SOFTMAX, "sigmoid": rt.HEAD_SIGMOID}[self.head.act_func]
        lin = self.head.classifier[1]
        plan.head([c[0] for c in cur], lin.weight, lin.bias, act)


# ================================================================================================ MobileNetV2
class MBInvertedResidual(_Holder):
    """mobilenetv2_helper.py:30-68 (class name `InvertedResidual` in the reference's module)."""

    def __init__(self, inp, oup, stride, expand_ratio):
        super().__init__()
        self.stride = stride
        hidden_dim = round(inp * expand_ratio)
        self.use_res_connect = self.stride == (1, 1, 1) and inp == oup
        if expand_ratio == 1:
            self.conv = nn.Sequential(
                nn.Conv3d(hidden_dim, hidden_dim, 3, stride, 1, groups=hidden_dim, bias=False),
                nn.BatchNorm3d(hidden_dim), nn.ReLU6(inplace=True),
                nn.Conv3d(hidden_dim, oup, 1, 1, 0, bias=False), nn.BatchNorm3d(oup))
        else:
            self.conv = nn.Sequential(
                nn.Conv3d(inp, hidden_dim, 1, 1, 0, bias=False), nn.BatchNorm3d(hidden_dim), nn.ReLU6(inplace=True),
                nn.Conv3d(hidden_dim, hidden_dim, 3, stride, 1, groups=hidden_dim, bias=False),
                nn.BatchNorm3d(hidden_dim), nn.ReLU6(inplace=True),
                nn.Conv3d(hidden_dim, oup, 1, 1, 0, bias=False), nn.BatchNorm3d(oup))


class MobileV2_Inverted_Residual_Block(_Holder):
    """mobilenetv2_helper.py:71-105."""

    def __init__(self, input_channel, setting, width_mult, beta_inv=None):
        super().__init__()
        feats = []
        rows = setting if isinstance(setting[0], list) else [setting]
        for t, c, n, s in rows:
            output_channel = int(c * width_mult) if beta_inv is None else int(c * width_mult // beta_inv)
            for i in range(n):
                feats.append(MBInvertedResidual(input_channel, output_channel, s if i == 0 else (1, 1, 1), t))
                input_channel = output_channel
        self.features = nn.Sequential(*feats)


class MobileNetV2_Stage(_Holder):
    """mobilenetv2_helper.py:258-343."""

    def __init__(self, input_channel, slow_residual_setting, fast_residual_setting, width_mult=1.0, beta_inv=4):
        super().__init__()
        self.names = []
        for p, (setting, binv) in enumerate(((slow_residual_setting, None), (fast_residual_setting, beta_inv))):
            blk = MobileV2_Inverted_Residual_Block(input_channel[p], setting, width_mult, beta_inv=binv)
            name = "pathway{}_channel_{}".format(p, setting[0][1])
            self.add_module(name, blk)
            self.names.append(name)
            _stage_init(self)

    def pathway(self, p):
        return getattr(self, self.names[p])


class MobilenetV2_Basic_Stem(_Holder):
    """stem_helper.py:191-201."""

    def __init__(self, input_channel, width_mult, img_dim):
        super().__init__()
        c = int(input_channel * width_mult)
        self.features = nn.Sequential(
            nn.Conv3d(img_dim, c, kernel_size=3, stride=(1, 2, 2), padding=(1, 1, 1), bias=False), nn.BatchNorm3d(c),
            nn.ReLU6(inplace=True))


class MobilenetV2_Model_Stem(_Holder):
    """stem_helper.py:204-232."""

    def __init__(self, input_channels, width_mult, img_dim=3):
        super().__init__()
        self.num_pathways = len(input_channels)
        for p in range(self.num_pathways):
            self.add_module("pathway{}_stem".format(p), MobilenetV2_Basic_Stem(input_channels[p], width_mult[p], img_dim))


class MobileNetV2BasicHead(_Holder):
    """head_helper.py:436-486: per pathway 1x1x1 conv + BN + ReLU6 -> global avg -> cat -> Dropout -> Linear -> softmax."""

    def __init__(self, input_channel, last_channel, num_classes, dropout_rate, act_func="softmax"):
        super().__init__()
        self.num_pathways = len(input_channel)
        for p in range(self.num_pathways):
            feats = nn.Sequential(nn.Conv3d(input_channel[p], last_channel[p], kernel_size=1, stride=1, padding=0,
                                            bias=False), nn.BatchNorm3d(last_channel[p]), nn.ReLU6(inplace=True))
            self.add_module("pathway{}_conv1x1x1".format(p), feats)
        if act_func == "softmax":
            self.act = nn.Softmax(dim=4)
        elif act_func == "sigmoid":
            self.act = nn.Sigmoid()
        self.act_func = act_func
        self.classifier = nn.Sequential(nn.Dropout(dropout_rate), nn.Linear(sum(last_channel), num_classes, bias=True))


_MBV2_SETTING = [  # custom_video_model_builder.py:1029-1047 (t, c, n, s), identical for both pathways
    [1, 16, 1, (1, 1, 1)], [6, 24, 2, (1, 2, 2)], [6, 32, 3, (1, 2, 2)], [6, 64, 4, (1, 2, 2)],
    [6, 96, 3, (1, 1, 1)], [6, 160, 3, (1, 2, 2)], [6, 320, 1, (1, 1, 1)]]


@MODEL_REGISTRY.register()
class SlowFastMoibleNetV2(_EfficientBase):
    """custom_video_model_builder.py:1057-1285 (the class name is spelled this way in the reference)."""

    def __init__(self, cfg):
        super().__init__()
        self.norm_module = get_norm(cfg)
        if cfg.DETECTION.ENABLE:
            raise NotImplementedError("DETECTION.ENABLE is out of scope")
        self.enable_detection = False
        wm, beta, alpha = cfg.SLOWFAST.WIDTH_MULTI, cfg.SLOWFAST.BETA_INV, cfg.SLOWFAST.ALPHA
        L = _MBV2_SETTING
        wpg = 32
        self.last_channel = int(1280 * wm) if wm > 1.0 else 1280
        self.s1 = MobilenetV2_Model_Stem(input_channels=[wpg, wpg], width_mult=[wm, wm / beta],
                                         img_dim=len(cfg.DATA.MEAN))

        def stage(cin, rows):
            return MobileNetV2_Stage(input_channel=cin, slow_residual_setting=rows, fast_residual_setting=rows,
                                     width_mult=wm, beta_inv=beta)

        def fuse(c):
            return FuseFastAndSlow(dim_in=[int(c * wm), int(c * wm) // beta], alpha=alpha, beta_inv=beta,
                                   norm_module=self.norm_module)

        def fused_in(c):   # input channels of the stage that follows a fusion of width c (reference arithmetic kept)
            return [int(c * wm + c * wm // beta), int(c * wm // beta + c * wm // beta)]

        self.s2 = stage([int(wpg * wm), int(wpg * wm // beta)], L[0:2])
        self.s3_fuse = fuse(L[1][1])
        self.s4 = stage(fused_in(L[1][1]), L[2:3])
        self.s4_fuse = fuse(L[2][1])
        self.s5 = stage(fused_in(L[2][1]), L[3:4])
        self.s5_fuse = fuse(L[3][1])
        self.s6 = stage(fused_in(L[3][1]), L[4:5])
        self.s7 = stage([int(L[4][1] * wm), int(L[4][1] * wm // beta)], L[5:6])
        self.s7_fuse = fuse(L[5][1])
        self.s8 = stage(fused_in(L[5][1]), L[6:])
        self.head = MobileNetV2BasicHead(
            input_channel=[int(L[6][1] * wm), int(L[6][1] * wm // beta)],
            last_channel=[self.last_channel, self.last_channel // beta], num_classes=cfg.MODEL.NUM_CLASSES,
            dropout_rate=cfg.MODEL.DROPOUT_RATE, act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    def _emit_unit(self, plan, unit, x, y):
        """InvertedResidual.forward (mobilenetv2_helper.py:64-68)."""
        seq = unit.conv
        res = x if unit.use_res_connect else None
        if len(seq) == 5:    # expand_ratio == 1: dw + BN + ReLU6 -> pw-linear + BN
            t = self._emit_conv(plan, x, seq[0], seq[1], rt.ACT_RELU6)
            self._emit_conv(plan, t, seq[3], seq[4], rt.ACT_NONE, y=y, res=res)
        else:
            t = self._emit_conv(plan, x, seq[0], seq[1], rt.ACT_RELU6)
            t = self._emit_conv(plan, t, seq[3], seq[4], rt.ACT_RELU6)
            self._emit_conv(plan, t, seq[6], seq[7], rt.ACT_NONE, y=y, res=res)

    def _emit_stage(self, plan, stage, cur, fuse_after, name):
        """Runs both pathways of a stage.  `cur` entries are plain tensors (whole buffers).  When a fusion follows,
        the last unit writes into its slice of the fusion's concat buffer."""
        beta = self._cfg.SLOWFAST.BETA_INV
        B = cur[0].shape[0]
        outs = []
        for p in range(2):
            x = cur[p]
            units = stage.pathway(p).features
            c_own = units[-1].conv[-2].out_channels
            _, T, H, W, _ = x.shape
            for u in units:
                s = u.stride
                H, W = _conv_out(H, 3, s[1], 1), _conv_out(W, 3, s[2], 1)
            outs.append((c_own, T, H, W))
        bufs = []
        for p in range(2):
            c_own, T, H, W = outs[p]
            if fuse_after:
                cs, cf = outs[0][0], outs[1][0]
                tot = cs + cf if p == 0 else cs // beta + cf
                off = 0 if p == 0 else cs // beta
            else:
                tot, off = c_own, 0
            bufs.append((plan.act(B, T, H, W, tot, name="%s_cat%d" % (name, p)), off, c_own))
        for p in range(2):
            x = cur[p]
            units = stage.pathway(p).features
            dst, off, c_own = bufs[p]
            _, T, H, W, _ = x.shape
            for ui, u in enumerate(units):
                s = u.stride
                H, W = _conv_out(H, 3, s[1], 1), _conv_out(W, 3, s[2], 1)
                last = ui == len(units) - 1
                y = dst[..., off:off + c_own] if last else plan.act(B, T, H, W, u.conv[-2].out_channels)
                self._emit_unit(plan, u, x, y)
                x = y
        return bufs

    def _compile(self, plan):
        cfg = self._cfg
        alpha = cfg.SLOWFAST.ALPHA
        xs_in = plan.inputs
        B = xs_in[0].shape[0]
        assert xs_in[1].shape[2] == xs_in[0].shape[2] * alpha, "fast pathway must have ALPHA x the frames of the slow one"
        cur = []
        for p in range(2):
            seq = getattr(self.s1, "pathway{}_stem".format(p)).features
            _, _, T, H, W = xs_in[p].shape
            T, H, W = self._pooled_shape(T, H, W, seq)
            buf = plan.act(B, T, H, W, seq[0].out_channels, name="s1_cat%d" % p)
            w, b = plan.once(fold_conv_bn, seq[0].weight, None, seq[1])
            plan.stem(xs_in[p], buf, w, b, tuple(seq[0].stride), tuple(seq[0].padding), act=rt.ACT_RELU6)
            cur.append(buf)
        order = [("s2", True, "s3_fuse"), ("s4", True, "s4_fuse"), ("s5", True, "s5_fuse"), ("s6", False, None),
                 ("s7", True, "s7_fuse"), ("s8", False, None)]
        for sname, fuse_after, fname in order:
            bufs = self._emit_stage(plan, getattr(self, sname), cur, fuse_after, sname)
            if fuse_after:
                self._emit_fuse(plan, getattr(self, fname), bufs)
            cur = [b[0] for b in bufs]
        feats = []
        for p in range(2):
            seq = getattr(self.head, "pathway{}_conv1x1x1".format(p))
            feats.append(self._emit_conv(plan, cur[p], seq[0], seq[1], rt.ACT_RELU6))
        act = {"softmax": rt.HEAD_SOFTMAX, "sigmoid": rt.HEAD_SIGMOID}[self.head.act_func]
        lin = self.head.classifier[1]
        plan.head(feats, lin.weight, lin.bias, act)


MODEL_REGISTRY.register(SlowFastMoibleNetV2, name="SlowFastMobileNetV2")   # BASELINE.json spelling


# ================================================================================================ GhostNet
def _make_divisible(v, divisor, min_value=None):
    """ghostnet_helper.py:11-24."""
    if min_value is None:
        min_value = divisor
    new_v = max(min_value, int(v + divisor / 2) // divisor * divisor)
    if new_v < 0.9 * v:
        new_v += divisor
    return new_v


class SqueezeExcite(_Holder):
    """ghostnet_helper.py:34-52 (gate: hard sigmoid)."""

    def __init__(self, in_chs, se_ratio=0.25, divisor=4):
        super().__init__()
        reduced_chs = _make_divisible(in_chs * se_ratio, divisor)
        self.avg_pool = nn.AdaptiveAvgPool3d(1)
        self.conv_reduce = nn.Conv3d(in_chs, reduced_chs, 1, bias=True)
        self.act1 = nn.ReLU(inplace=True)
        self.conv_expand = nn.Conv3d(reduced_chs, in_chs, 1, bias=True)


class ConvBnAct(_Holder):
    """ghostnet_helper.py:55-68 / head_helper.py:612-627."""

    def __init__(self, in_chs, out_chs, kernel_size, stride=1):
        super().__init__()
        self.conv = nn.Conv3d(in_chs, out_chs, kernel_size, stride, kernel_size // 2, bias=False)
        self.bn1 = nn.BatchNorm3d(out_chs)
        self.act1 = nn.ReLU(inplace=True)


class GhostModule(_Holder):
    """ghostnet_helper.py:71-99: 1xkxk primary conv + depthwise 3x3x3 'cheap operation', concat, slice to `oup`."""

    def __init__(self, inp, oup, kernel_size=1, ratio=2, dw_size=3, stride=1, relu=True):
        super().__init__()
        self.oup = oup
        self.relu = relu
        init_channels = math.ceil(oup / ratio)
        new_channels = init_channels * (ratio - 1)
        self.primary_conv = nn.Sequential(
            nn.Conv3d(inp, init_channels, kernel_size=(1, kernel_size, kernel_size), stride=(1, stride, stride),
                      padding=(0, kernel_size // 2, kernel_size // 2), bias=False),
            nn.BatchNorm3d(init_channels), nn.ReLU(inplace=True) if relu else nn.Sequential())
        self.cheap_operation = nn.Sequential(
            nn.Conv3d(init_channels, new_channels, kernel_size=dw_size, stride=1, padding=dw_size // 2,
                      groups=init_channels, bias=False),
            nn.BatchNorm3d(new_channels), nn.ReLU(inplace=True) if relu else nn.Sequential())


class GhostBottleneck(_Holder):
    """ghostnet_helper.py:102-163."""

    def __init__(self, in_chs, mid_chs, out_chs, dw_kernel_size=3, stride=1, se_ratio=0.0):
        super().__init__()
        has_se = se_ratio is not None and se_ratio > 0.0
        self.stride = stride
        self.ghost1 = GhostModule(in_chs, mid_chs, relu=True)
        if self.stride > 1:
            self.conv_dw = nn.Conv3d(mid_chs, mid_chs, kernel_size=(1, dw_kernel_size, dw_kernel_size),
                                     stride=(1, stride, stride),
                                     padding=(0, (dw_kernel_size - 1) // 2, (dw_kernel_size - 1) // 2), groups=mid_chs,
                                     bias=False)
            self.bn_dw = nn.BatchNorm3d(mid_chs)
        self.se = SqueezeExcite(mid_chs, se_ratio=se_ratio) if has_se else None
        self.ghost2 = GhostModule(mid_chs, out_chs, relu=False)
        if in_chs == out_chs and self.stride == 1:
            self.shortcut = nn.Sequential()
        else:
            self.shortcut = nn.Sequential(
                nn.Conv3d(in_chs, in_chs, kernel_size=(1, dw_kernel_size, dw_kernel_size), stride=(1, stride, stride),
                          padding=(0, (dw_kernel_size - 1) // 2, (dw_kernel_size - 1) // 2), groups=in_chs, bias=False),
                nn.BatchNorm3d(in_chs), nn.Conv3d(in_chs, out_chs, 1, stride=1, padding=0, bias=False),
                nn.BatchNorm3d(out_chs))


class GhostNet_Inverted_Residual_Block(_Holder):
    """ghostnet_helper.py:266-312."""

    def __init__(self, input_channel, cfg):
        super().__init__()
        layers = []
        for k, exp_size, c, se_ratio, s in cfg:
            output_channel = _make_divisible(c, 2)
            hidden_channel = _make_divisible(exp_size, 2)
            layers.append(GhostBottleneck(input_channel, hidden_channel, output_channel, dw_kernel_size=k, stride=s,
                                          se_ratio=se_ratio))
            input_channel = output_channel
        self.features = nn.Sequential(*layers)
        _stage_init(self)


class GhostNet_Stage(_Holder):
    """ghostnet_helper.py:315-380."""

    def __init__(self, input_channel, slow_cfg, fast_cfg):
        super().__init__()
        self.names = []
        for p, cfg in enumerate((slow_cfg, fast_cfg)):
            name = "pathway{}_channel_{}".format(p, cfg[-1][2])
            self.add_module(name, GhostNet_Inverted_Residual_Block(input_channel[p], cfg))
            self.names.append(name)
            _stage_init(self)

    def pathway(self, p):
        return getattr(self, self.names[p])


class GhostNet_Model_Stem(_Holder):
    """stem_helper.py:310-336: Conv3d 3x3x3 s(1,2,2) p1 -> BN -> ReLU (no pool)."""

    def __init__(self, input_channels, img_dim=3):
        super().__init__()
        for p in range(len(input_channels)):
            self.add_module("pathway{}_stem".format(p), nn.Sequential(
                nn.Conv3d(img_dim, input_channels[p], kernel_size=3, stride=(1, 2, 2), padding=1, bias=False),
                nn.BatchNorm3d(input_channels[p]), nn.ReLU(inplace=True)))


class GhostNetBasicHead(_Holder):
    """head_helper.py:630-700.  `self.act` is overwritten with ReLU in the reference (:653), so the eval output is
    ReLU(logits), not a softmax -- reproduced."""

    def __init__(self, input_channel, mid_channel, output_channel, num_classes, dropout_rate, act_func="softmax"):
        super().__init__()
        self.num_pathways = len(input_channel)
        self.stage5_conv_slow = ConvBnAct(input_channel[0], mid_channel[0], 1)
        self.stage5_conv_fast = ConvBnAct(input_channel[1], mid_channel[1], 1)
        self.conv_head_slow = nn.Conv3d(mid_channel[0], output_channel[0], 1, 1, 0, bias=True)
        self.conv_head_fast = nn.Conv3d(mid_channel[1], output_channel[1], 1, 1, 0, bias=True)
        self.act = nn.ReLU(inplace=True)
        self.classifier = nn.Sequential(nn.Dropout(dropout_rate), nn.Linear(sum(output_channel), num_classes, bias=True))


_GHOST_STAGES = [   # k, t, c, SE, s   (custom_video_model_builder.py:813-845)
    [[3, 16, 16, 0, 1]],
    [[3, 48, 24, 0, 2], [3, 72, 24, 0, 1]],
    [[5, 72, 40, 0.25, 2], [5, 120, 40, 0.25, 1]],
    [[3, 240, 80, 0, 2], [3, 200, 80, 0, 1], [3, 184, 80, 0, 1], [3, 184, 80, 0, 1], [3, 480, 112, 0.25, 1],
     [3, 672, 112, 0.25, 1]],
    [[5, 672, 160, 0.25, 2], [5, 960, 160, 0, 1], [5, 960, 160, 0.25, 1], [5, 960, 160, 0, 1], [5, 960, 160, 0.25, 1]],
]


def ghost_cfgs(wm, beta):
    slow, fast = [], []
    for stage in _GHOST_STAGES:
        fast.append([[c[0], _make_divisible(c[1] * wm // beta, 4), _make_divisible(c[2] * wm // beta, 4), c[3], c[4]]
                     for c in stage])
        slow.append([[c[0], _make_divisible(c[1] * wm, 4), _make_divisible(c[2] * wm, 4), c[3], c[4]] for c in stage])
    return slow, fast


@MODEL_REGISTRY.register()
class SlowFastGhostNet(_EfficientBase):
    """custom_video_model_builder.py:792-1026."""

    def __init__(self, cfg):
        super().__init__()
        self.norm_module = get_norm(cfg)
        if cfg.DETECTION.ENABLE:
            raise NotImplementedError("DETECTION.ENABLE is out of scope")
        self.enable_detection = False
        wm, beta, alpha = cfg.SLOWFAST.WIDTH_MULTI, cfg.SLOWFAST.BETA_INV, cfg.SLOWFAST.ALPHA
        self.slow_cfgs, self.fast_cfgs = ghost_cfgs(wm, beta)
        sc, fc = self.slow_cfgs, self.fast_cfgs
        widths = [_make_divisible(16 * wm, 4), _make_divisible(16 * wm // beta, 4)]
        outs = [int(1280 * wm), int(1280 * wm // beta)]
        self.s0 = GhostNet_Model_Stem(input_channels=widths, img_dim=len(cfg.DATA.MEAN))
        self.s1 = GhostNet_Stage(input_channel=widths, slow_cfg=sc[0], fast_cfg=fc[0])
        for i in range(4):
            fuse = FuseFastAndSlow(dim_in=[sc[i][-1][2], fc[i][-1][2]], alpha=alpha, beta_inv=beta,
                                   norm_module=self.norm_module)
            setattr(self, "s%d_fuse" % (i + 1), fuse)
            own_s = sc[i][0][2] if i < 3 else sc[i][-1][2]      # the reference indexes [0][2] for s2..s4, [-1][2] for s5
            own_f = fc[i][0][2] if i < 3 else fc[i][-1][2]
            stage = GhostNet_Stage(input_channel=[own_s + fc[i][-1][2], own_f + sc[i][-1][2] // beta],
                                   slow_cfg=sc[i + 1], fast_cfg=fc[i + 1])
            setattr(self, "s%d" % (i + 2), stage)
        self.head = GhostNetBasicHead(input_channel=[sc[4][-1][2], fc[4][-1][2]], mid_channel=[sc[4][-1][1], fc[4][-1][1]],
                                      output_channel=outs, num_classes=cfg.MODEL.NUM_CLASSES,
                                      dropout_rate=cfg.MODEL.DROPOUT_RATE, act_func=cfg.MODEL.HEAD_ACT)
        init_weights(self, cfg.MODEL.FC_INIT_STD, cfg.RESNET.ZERO_INIT_FINAL_BN)
        self._init_runtime(cfg)

    def _emit_ghost(self, plan, gm, x, out, res=None):
        """GhostModule.forward (ghostnet_helper.py:95-99) into `out` (oup channels).  With `res` (ghost2 of a
        bottleneck) the residual is added after the concat; the cheap operation must read the un-added primary
        output, so that goes through a temporary."""
        act = rt.ACT_RELU if gm.relu else rt.ACT_NONE
        pc, pbn = gm.primary_conv[0], gm.primary_conv[1]
        cc, cbn = gm.cheap_operation[0], gm.cheap_operation[1]
        init = pc.out_channels
        keep = gm.oup - init                                  # channels of the cheap branch that survive the slice
        B, T, H, W, _ = out.shape
        x1 = out[..., :init] if res is None else plan.act(B, T, H, W, init)
        self._emit_conv(plan, x, pc, pbn, act, y=x1)
        if keep > 0:
            w, b = plan.once(fold_conv_bn, cc.weight, cc.bias, cbn)
            # depthwise with channel multiplier 1: output channel j reads input channel j -> truncating is exact
            plan.conv(x1[..., :keep], out[..., init:init + keep], w[:keep], b[:keep], stride=tuple(cc.stride),
                      padding=tuple(cc.padding), groups=keep, act=act, res=None if res is None else res[..., init:init + keep])
        if res is not None:
            plan.eltwise_add(x1, res[..., :init], out[..., :init])

    def _emit_unit(self, plan, blk, x, y):
        """GhostBottleneck.forward (ghostnet_helper.py:149-163)."""
        B, T, H, W, _ = x.shape
        mid = blk.ghost1.oup
        g1 = plan.act(B, T, H, W, mid)
        self._emit_ghost(plan, blk.ghost1, x, g1)
        t = g1
        if blk.stride > 1:
            t = self._emit_conv(plan, t, blk.conv_dw, blk.bn_dw, rt.ACT_NONE)
        if blk.se is not None:
            t2 = plan.act(*t.shape)
            plan.squeeze_excite(t, t2, blk.se)
            t = t2
        if len(blk.shortcut) == 0:
            sc = x
        else:
            sc = self._emit_conv(plan, x, blk.shortcut[0], blk.shortcut[1], rt.ACT_NONE)
            sc = self._emit_conv(plan, sc, blk.shortcut[2], blk.shortcut[3], rt.ACT_NONE)
        self._emit_ghost(plan, blk.ghost2, t, y, res=sc)

    def _emit_stage(self, plan, stage, cur, fuse_after, name):
        beta = self._cfg.SLOWFAST.BETA_INV
        B = cur[0].shape[0]
        outs = []
        for p in range(2):
            units = stage.pathway(p).features
            _, T, H, W, _ = cur[p].shape
            for u in units:
                if u.stride > 1:
                    k = u.conv_dw.kernel_size[1]
                    H, W = _conv_out(H, k, u.stride, (k - 1) // 2), _conv_out(W, k, u.stride, (k - 1) // 2)
            outs.append((units[-1].ghost2.oup, T, H, W))
        bufs = []
        for p in range(2):
            c_own, T, H, W = outs[p]
            if fuse_after:
                cs, cf = outs[0][0], outs[1][0]
                tot = cs + cf if p == 0 else cs // beta + cf
                off = 0 if p == 0 else cs // beta
            else:
                tot, off = c_own, 0
            bufs.append((plan.act(B, T, H, W, tot, name="%s_cat%d" % (name, p)), off, c_own))
        for p in range(2):
            x = cur[p]
            units = stage.pathway(p).features
            dst, off, c_own = bufs[p]
            _, T, H, W, _ = x.shape
            for ui, u in enumerate(units):
                if u.stride > 1:
                    k = u.conv_dw.kernel_size[1]
                    H, W = _conv_out(H, k, u.stride, (k - 1) // 2), _conv_out(W, k, u.stride, (k - 1) // 2)
                last = ui == len(units) - 1
                y = dst[..., off:off + c_own] if last else plan.act(B, T, H, W, u.ghost2.oup)
                self._emit_unit(plan, u, x, y)
                x = y
        return bufs

    def _compile(self, plan):
        cfg = self._cfg
        alpha = cfg.SLOWFAST.ALPHA
        xs_in = plan.inputs
        B = xs_in[0].shape[0]
        assert xs_in[1].shape[2] == xs_in[0].shape[2] * alpha, "fast pathway must have ALPHA x the frames of the slow one"
        cur = []
        for p in range(2):
            seq = getattr(self.s0, "pathway{}_stem".format(p))
            _, _, T, H, W = xs_in[p].shape
            T, H, W = self._pooled_shape(T, H, W, seq)
            buf = plan.act(B, T, H, W, seq[0].out_channels, name="s0_cat%d" % p)
            w, b = plan.once(fold_conv_bn, seq[0].weight, None, seq[1])
            plan.stem(xs_in[p], buf, w, b, tuple(seq[0].stride), tuple(seq[0].padding), act=rt.ACT_RELU)
            cur.append(buf)
        for i in range(1, 6):
            fuse_after = i < 5
            bufs = self._emit_stage(plan, getattr(self, "s%d" % i), cur, fuse_after, "s%d" % i)
            if fuse_after:
                self._emit_fuse(plan, getattr(self, "s%d_fuse" % i), bufs)
            cur = [b[0] for b in bufs]
        h = self.head
        outs = [h.conv_head_slow.out_channels, h.conv_head_fast.out_channels]
        feat = plan.alloc((B, sum(outs)), torch.float32)
        col = 0
        for p, (cba, ch) in enumerate(((h.stage5_conv_slow, h.conv_head_slow), (h.stage5_conv_fast, h.conv_head_fast))):
            t = self._emit_conv(plan, cur[p], cba.conv, cba.bn1, rt.ACT_RELU)
            plan.pooled_fc(t, ch.weight, ch.bias, rt.HEAD_RELU, feat[:, col:], sum(outs))
            col += outs[p]
        lin = h.classifier[1]
        plan.fc(feat, lin.weight, lin.bias, rt.HEAD_RELU)   # eval "act" of this head is ReLU (head_helper.py:653)
