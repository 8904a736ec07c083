"""AVA detection on the GPU: the RoI-head kernels (esf_temporal_mean, esf_roi_align_max) against torchvision's
roi_align, and forward(x, bboxes) of the SlowFast / Slow R50 detection models against the CPU detection oracle.

The models reuse the calibrated BN statistics of the slowfast_r50 / slow_r50 golden fixtures: a detection model has the
same trunk BN keys as its classification counterpart (dilation changes no shape)."""
import ctypes

import pytest
import torch

import detection_oracle as DO
import helpers
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.workloads import seeded_state_dict
from oracle import input_oracle as IO

pytestmark = pytest.mark.gpu
BF16_TOL = 2e-2


# ------------------------------------------------------------------------------------------------ kernels
def _boxes(K, B, H_px, W_px, seed):
    """K boxes over B clips, batch indices unsorted, sizes from a few pixels to beyond the frame."""
    g = torch.Generator().manual_seed(seed)
    b = torch.randint(0, B, (K,), generator=g).float()
    cx, cy = torch.rand(K, generator=g) * W_px, torch.rand(K, generator=g) * H_px
    w = torch.rand(K, generator=g) * W_px * 1.2 + 2
    h = torch.rand(K, generator=g) * H_px * 1.2 + 2
    return torch.stack([b, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)


def _kernel_case(B, T, H, W, C, K, aligned, dtype, seed=0):
    from torchvision.ops import roi_align

    L = rt.lib()
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, H, W, C, generator=g).to(dtype).cuda()
    boxes = _boxes(K, B, H * 16, W * 16, seed + 1)
    m = torch.empty(B, H, W, C, dtype=torch.float32, device="cuda")
    feat = torch.full((K, C + 8), -7.0, device="cuda")
    xv = rt.view(x)
    s = rt.current_stream_ptr()
    rt.check(L.esf_temporal_mean(ctypes.byref(xv), m.data_ptr(), s), "esf_temporal_mean")
    bd = boxes.cuda()
    rt.check(L.esf_roi_align_max(m.data_ptr(), B, H, W, C, bd.data_ptr(), K, 1.0 / 16, 7, int(aligned),
                                 feat.data_ptr(), C + 8, 8, s), "esf_roi_align_max")
    torch.cuda.synchronize()
    mean_ref = x.float().mean(1)
    assert helpers.rel_err(m.cpu(), mean_ref.cpu()) <= 1e-6
    ref = roi_align(m.permute(0, 3, 1, 2).cpu(), boxes, 7, 1.0 / 16, 0, aligned).amax(dim=(2, 3))
    got = feat.cpu()
    assert torch.equal(got[:, :8], torch.full((K, 8), -7.0))      # the slice before c_off is left alone
    err = helpers.rel_err(got[:, 8:], ref)
    print("roi B%d %dx%d C%d K%d aligned=%s: rel err %.2e" % (B, H, W, C, K, aligned, err))
    assert err <= 1e-5


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("C,H,W,K,B", [(2048, 14, 20, 1, 1), (2048, 16, 22, 300, 4), (256, 14, 14, 300, 3),
                                       (256, 9, 13, 1, 2)])
def test_roi_kernels_match_torchvision(esf_lib, C, H, W, K, B, aligned):
    _kernel_case(B, 8, H, W, C, K, aligned, torch.float16)


def test_roi_kernels_bf16_and_odd_channels(esf_lib):
    _kernel_case(2, 4, 7, 11, 2048, 40, True, torch.bfloat16)
    _kernel_case(2, 3, 7, 11, 100, 40, False, torch.float16)     # C % 8 != 0: the scalar temporal mean


# ------------------------------------------------------------------------------------------------ models
def _detection_model(name, precision="fp16"):
    """slowfast_r50 / slow_r50 with the AVA head: DETECTION.ENABLE, res5 at stride 1 and dilation 2, 80 sigmoid
    classes; seeded weights with the fixture's calibrated BN statistics."""
    cfg = helpers.case_cfg(name)
    npw = len(cfg.DATA.INPUT_CHANNEL_NUM)
    cfg.RESNET.SPATIAL_STRIDES = [[1] * npw, [2] * npw, [2] * npw, [1] * npw]
    cfg.RESNET.SPATIAL_DILATIONS = [[1] * npw, [1] * npw, [1] * npw, [2] * npw]
    cfg.DETECTION.ENABLE = True
    cfg.MODEL.NUM_CLASSES, cfg.MODEL.HEAD_ACT = 80, "sigmoid"
    cfg.MULTIGRID.SHORT_CYCLE = False
    cfg.ESF.PRECISION = precision
    from efficient_slowfast_b200 import build_model

    torch.manual_seed(0)
    model = build_model(cfg)
    gold = helpers.load_golden(name)
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    model.load_state_dict(seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    return cfg, model.eval()


def _clip(cfg, B, H, W, seed=3):
    g = torch.Generator().manual_seed(seed)
    fast = torch.randn(B, 3, cfg.DATA.NUM_FRAMES, H, W, generator=g)
    if len(cfg.DATA.INPUT_CHANNEL_NUM) == 1:
        return [fast]
    idx = torch.linspace(0, fast.shape[2] - 1, fast.shape[2] // cfg.SLOWFAST.ALPHA).long()
    return [fast.index_select(2, idx).contiguous(), fast]


CASES = [("slowfast_r50", 64, 64), ("slowfast_r50", 64, 96), ("slow_r50", 64, 64), ("slow_r50", 64, 96)]


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("name,H,W", CASES)
def test_detection_model_matches_oracle(esf_lib, name, H, W, precision):
    cfg, model = _detection_model(name, precision)
    xs = _clip(cfg, 2, H, W)
    boxes = _boxes(11, 2, H, W, seed=5)
    want = DO.forward(cfg, model.state_dict(), xs, boxes)
    model = model.cuda()
    with torch.no_grad():
        y = model([t.cuda() for t in xs], boxes).cpu()
    err = helpers.rel_err(y, want)
    tol = BF16_TOL if precision == "fp16" else 6e-2
    print("%s %dx%d %s: rel err %.3e (tol %.0e)" % (name, H, W, precision, err, tol))
    assert y.shape == (11, 80) and y.dtype == torch.float32
    assert err <= tol


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_detection_forward_paths_and_box_sets_agree(esf_lib, name):
    """Bit-exact: forward / forward_fast / forward_frames; CUDA graph on and off; permuted and subset boxes give the
    same rows; the box count never creates a second plan; K = 0 is an empty result."""
    cfg, model = _detection_model(name)
    model = model.cuda()
    two = model.num_pathways == 2
    g = torch.Generator().manual_seed(12)
    fr = torch.randint(0, 256, (2, cfg.DATA.NUM_FRAMES, 64, 96, 3), generator=g, dtype=torch.uint8)
    xs = IO.frames_to_inputs(fr, cfg.DATA.MEAN, cfg.DATA.STD, cfg.SLOWFAST.ALPHA if two else 1, not two, False)
    xs = [t.cuda() for t in xs]
    boxes = _boxes(23, 2, 64, 96, seed=9)
    with torch.no_grad():
        y = model(xs, boxes).cpu()
        assert torch.isfinite(y).all()
        assert torch.equal(model.forward_frames(fr.cuda(), boxes).cpu(), y)
        if two:
            assert torch.equal(model.forward_fast(xs[1], boxes).cpu(), y)
        assert torch.equal(model(xs, boxes.cuda()).cpu(), y)                      # device boxes
        perm = torch.randperm(23, generator=g)
        assert torch.equal(model(xs, boxes[perm]).cpu(), y[perm])
        sub = torch.tensor([17, 2, 5])
        assert torch.equal(model(xs, boxes[sub]).cpu(), y[sub])
        assert torch.equal(model(xs, boxes[:1]).cpu(), y[:1])
        big = torch.cat([boxes] * 20)                                             # K = 460: the buffers grow
        assert torch.equal(model(xs, big).cpu(), torch.cat([y] * 20))
        empty = model(xs, boxes[:0])
        assert empty.shape == (0, 80) and empty.device.type == "cuda"
        assert len(model._plans) == 1
        cfg.ESF.CUDA_GRAPH = False
        eager = model.__class__(cfg).cuda().eval()
        eager.load_state_dict(model.state_dict())
        assert not eager._use_graph
        assert torch.equal(eager(xs, boxes).cpu(), y)
        with pytest.raises(ValueError):
            model(xs)                                                            # a detection model needs boxes
        with pytest.raises(ValueError):
            model(xs, torch.tensor([[2.0, 0, 0, 10, 10]]))                       # batch index outside [0, 2)
