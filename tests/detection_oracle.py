"""TEST INFRASTRUCTURE ONLY -- CPU oracle of the AVA detection forward (SlowFast / ResNet with ResNetRoIHead).

Restates, with torch CPU ops on a reference-schema state_dict:
  * torchvision's `roi_align` (ops/csrc/ops/cpu/roi_align_kernel.cpp), which detectron2's `ROIAlign` dispatches to;
  * `ResNetRoIHead.forward` (SlowFast/slowfast/models/head_helper.py:100-130);
  * the detection branches of `SlowFast.forward` / `ResNet.forward` (video_model_builder.py): the trunk of the
    classification oracle's own forwards, then the RoI head on `bboxes`.
The classification oracle (oracle/slowfast_oracle.py) is pinned to the reference-made golden fixtures and stays
unchanged; this module only adds the head.
"""
import torch
import torch.nn.functional as F

from oracle import slowfast_oracle as O


def roi_align(x, boxes, output_size, spatial_scale, sampling_ratio=0, aligned=True):
    """torchvision.ops.roi_align(x, boxes, output_size, spatial_scale, sampling_ratio, aligned): x (N, C, H, W),
    boxes (K, 5) rows [batch index, x1, y1, x2, y2] -> (K, C, R, R).  Per bin: the mean of a grid_h x grid_w grid of
    bilinear samples (grid = sampling_ratio, or ceil(roi extent / R) when 0), taps outside [-1, H] x [-1, W] count as 0,
    the others are clamped to the map; `aligned` shifts the box by -0.5 cell and drops the legacy 1 x 1 minimum size.
    Box geometry, tap weights and the per-bin sum are computed in x.dtype in torchvision's order of operations (the
    samples of a bin are accumulated one after the other, iy outer, ix inner), so the result is torchvision's to the bit
    on the CPU."""
    N, C, H, W = x.shape
    R = int(output_size)
    dt = x.dtype
    bx = boxes.to(dt)
    K = bx.shape[0]
    out = x.new_zeros((K, C, R, R))
    off = 0.5 if aligned else 0.0
    scale = torch.tensor(spatial_scale, dtype=dt)
    p = torch.arange(R, dtype=dt)

    def axis(v, n):
        """bilinear_interpolate of torchvision along one axis: validity, low / high index, weights (l, 1 - l)."""
        valid = ~((v < -1.0) | (v > n))
        v = torch.where(v <= 0, torch.zeros_like(v), v)
        lo = v.floor().long()
        top = lo >= n - 1
        lo = torch.where(top, torch.full_like(lo, n - 1), lo)
        hi = torch.where(top, lo, lo + 1)
        v = torch.where(top, lo.to(dt), v)
        lv = v - lo.to(dt)
        return valid, lo.clamp(0, n - 1), hi.clamp(0, n - 1), lv, 1.0 - lv

    for k in range(K):
        b = int(bx[k, 0])
        sw, sh, ew, eh = (bx[k, 1] * scale - off, bx[k, 2] * scale - off, bx[k, 3] * scale - off, bx[k, 4] * scale - off)
        rw, rh = ew - sw, eh - sh
        if not aligned:
            rw, rh = torch.clamp_min(rw, 1.0), torch.clamp_min(rh, 1.0)
        bin_h, bin_w = rh / R, rw / R
        gh = sampling_ratio if sampling_ratio > 0 else int(torch.ceil(rh / R))
        gw = sampling_ratio if sampling_ratio > 0 else int(torch.ceil(rw / R))
        count = max(gh * gw, 1)
        m = x[b]
        acc = x.new_zeros((C, R, R))
        for iy in range(gh):
            vy, y0, y1, ly, hy = axis(sh + p * bin_h + (iy + 0.5) * bin_h / gh, H)          # one sample row per bin row
            for ix in range(gw):
                vx, x0, x1, lx, hx = axis(sw + p * bin_w + (ix + 0.5) * bin_w / gw, W)
                v1, v2 = m[:, y0][:, :, x0], m[:, y0][:, :, x1]
                v3, v4 = m[:, y1][:, :, x0], m[:, y1][:, :, x1]
                val = ((hy[:, None] * hx[None, :]) * v1 + (hy[:, None] * lx[None, :]) * v2
                       + (ly[:, None] * hx[None, :]) * v3 + (ly[:, None] * lx[None, :]) * v4)
                acc = acc + val * (vy[:, None] & vx[None, :]).to(dt)
        out[k] = acc / count
    return out


def resnet_roi_head(xs, sd, p, tpool, resolution, scale_factor, aligned, act, bboxes):
    """ResNetRoIHead.forward (head_helper.py:100-130): per pathway AvgPool3d([t, 1, 1], stride 1) (the pooled time axis
    must be 1), ROIAlign(R, 1 / scale, 0, aligned), MaxPool2d(R, stride 1); concat -> Linear -> softmax(dim 1) / sigmoid."""
    pooled = []
    for x, kt in zip(xs, tpool):
        out = F.avg_pool3d(x, [kt, 1, 1], stride=1)
        assert out.shape[2] == 1
        out = roi_align(out.squeeze(2), bboxes, resolution, 1.0 / scale_factor, 0, aligned)
        pooled.append(F.max_pool2d(out, resolution, stride=1))
    x = torch.cat(pooled, 1).reshape(bboxes.shape[0], -1)
    x = F.linear(x, sd[p + ".projection.weight"].to(x.dtype), sd[p + ".projection.bias"].to(x.dtype))
    if act == "softmax":
        return torch.softmax(x, dim=1)
    if act == "sigmoid":
        return torch.sigmoid(x)
    raise NotImplementedError(act)


def trunk(cfg, sd, inputs, dtype=torch.float32):
    """res5 outputs [slow, fast] (SlowFast) or [x] (ResNet) of the detection model, NCDHW: the classification oracle's
    own forward (oracle/slowfast_oracle.py), read at its "s5" tap.  Its classification head runs on a pool that fits
    any map -- global (MULTIGRID.SHORT_CYCLE) for SlowFast, a 1 x 1 spatial kernel (CROP_SIZE 32) for ResNet -- and its
    output is discarded."""
    c = cfg.clone()
    if c.MODEL.MODEL_NAME == "SlowFast":
        c.MULTIGRID.SHORT_CYCLE = True
    elif c.MODEL.MODEL_NAME == "ResNet":
        c.DATA.CROP_SIZE = 32
    else:
        raise NotImplementedError(c.MODEL.MODEL_NAME)
    taps = {}
    O.forward(c, sd, inputs, dtype=dtype, taps=taps)
    return taps["s5"]


def head(cfg, sd, xs, bboxes):
    """ResNetRoIHead of the detection model on res5 outputs `xs` (from trunk()): (K, NUM_CLASSES)."""
    nf, pool = cfg.DATA.NUM_FRAMES, O.POOL1[cfg.MODEL.ARCH]
    if len(xs) == 2:
        tpool = [nf // cfg.SLOWFAST.ALPHA // pool[0][0], nf // pool[1][0]]
    else:
        tpool = [nf // pool[0][0]]
    D = cfg.DETECTION
    sd = {k: v.detach().cpu() for k, v in sd.items() if k.startswith("head.")}
    with torch.no_grad():
        return resnet_roi_head(xs, sd, "head", tpool, D.ROI_XFORM_RESOLUTION, D.SPATIAL_SCALE_FACTOR, D.ALIGNED,
                               cfg.MODEL.HEAD_ACT, bboxes.detach().cpu().to(xs[0].dtype))


def forward(cfg, sd, inputs, bboxes, dtype=torch.float32):
    """Detection forward of cfg.MODEL.MODEL_NAME in ("SlowFast", "ResNet"): (K, NUM_CLASSES) for the (K, 5) boxes."""
    assert cfg.DETECTION.ENABLE
    return head(cfg, sd, trunk(cfg, sd, inputs, dtype), bboxes)
