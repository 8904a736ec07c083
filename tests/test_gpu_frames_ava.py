"""AVA detection from uint8 frames on the GPU: forward_ava_frames(frames, boxes) against forward(clips, bboxes) on what
the CPU restatement of the AVA test loader (tests/ava_frames_oracle.py) makes of the same frames and boxes, bit for bit,
for the SlowFast and Slow R50 detection models, both stem routes (packed 16-bit rows and the FP32 clip), landscape,
portrait and pure-window decode sizes, RGB and BGR; and the transformed boxes against the oracle's."""
import pytest
import torch

import ava_frames_oracle as AO
import helpers
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200.workloads import seeded_state_dict

pytestmark = pytest.mark.gpu

# (H0, W0, S): AVA's 256 x 340 (a pure window at 256), 4:3 and VGA (resized to 256 x 341), portrait, and small clips
# whose stems take the packed rows (64 x 96 is a pure window)
GEOMETRIES = [(256, 340, 256), (240, 320, 256), (480, 640, 256), (340, 256, 256), (64, 96, 64), (48, 80, 64),
              (120, 90, 112)]


def _model(name, precision="fp16", bgr=None):
    cfg = helpers.case_cfg(name)
    npw = len(cfg.DATA.INPUT_CHANNEL_NUM)
    cfg.RESNET.SPATIAL_STRIDES = [[1] * npw, [2] * npw, [2] * npw, [1] * npw]
    cfg.RESNET.SPATIAL_DILATIONS = [[1] * npw, [1] * npw, [1] * npw, [2] * npw]
    cfg.DETECTION.ENABLE = True
    cfg.MODEL.NUM_CLASSES, cfg.MODEL.HEAD_ACT = 80, "sigmoid"
    cfg.MULTIGRID.SHORT_CYCLE = False
    cfg.ESF.PRECISION = precision
    cfg.DATA.MEAN, cfg.DATA.STD = [0.45, 0.40, 0.35], [0.225, 0.25, 0.2]     # per-channel: the channel order shows
    if bgr is not None:
        cfg.AVA = cfg.DATA.__class__(dict(BGR=bgr))
    from efficient_slowfast_b200 import build_model

    torch.manual_seed(0)
    model = build_model(cfg)
    gold = helpers.load_golden(name)
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    model.load_state_dict(seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    return cfg, model.eval().cuda()


def _boxes(K, B, seed, dtype=torch.float64):
    """K loader boxes in [0, 1] (some crossing the edges) over B clips, batch indices unsorted."""
    g = torch.Generator().manual_seed(seed)
    b = torch.randint(0, B, (K,), generator=g).double()
    p = torch.rand(K, 4, generator=g, dtype=torch.float64) * 1.2 - 0.1
    x1, x2 = torch.minimum(p[:, 0], p[:, 2]), torch.maximum(p[:, 0], p[:, 2]) + 0.05
    y1, y2 = torch.minimum(p[:, 1], p[:, 3]), torch.maximum(p[:, 1], p[:, 3]) + 0.05
    return torch.stack([b, x1, y1, x2, y2], 1).to(dtype)


def _frames(cfg, B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, cfg.DATA.NUM_FRAMES, H, W, 3), generator=g, dtype=torch.uint8)


def _oracle(cfg, model, fr, boxes, S, bgr=False):
    two = model.num_pathways == 2
    return AO.prepare(fr, boxes, S, cfg.DATA.MEAN, cfg.DATA.STD, cfg.SLOWFAST.ALPHA if two else 1, not two, bgr,
                      bool(cfg.DATA.get("REVERSE_INPUT_CHANNEL", False)))


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_ava_frames_bit_identical_to_forward_on_oracle_clips(esf_lib, name):
    """Every geometry: scores, and the transformed boxes, equal forward(oracle clips, oracle boxes) bit for bit; both
    stem routes are covered by the geometries."""
    cfg, model = _model(name)
    routes = set()
    for i, (H, W, S) in enumerate(GEOMETRIES):
        fr = _frames(cfg, 2, H, W, seed=i)
        boxes = _boxes(9, 2, seed=30 + i)
        xs, want_boxes = _oracle(cfg, model, fr, boxes, S)
        with torch.no_grad():
            want = model([t.cuda() for t in xs], want_boxes.cuda()).cpu()
            got, px = model.forward_ava_frames(fr.cuda(), boxes, crop_size=S, return_boxes=True)
        plan = next(reversed(model._plans.values()))[1]
        routes |= {own.data_ptr() in plan.stem_routes for own in plan.inputs}
        print("%s %dx%d -> %s: packed stem rows %s" % (name, H, W, FR.resized_size(H, W, S),
                                                        [own.data_ptr() in plan.stem_routes for own in plan.inputs]))
        assert torch.isfinite(want).all()
        assert torch.equal(px.cpu(), want_boxes)
        assert torch.equal(got.cpu(), want)
    assert routes == {True, False}, "the geometries must cover both stem routes"


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_ava_frames_rgb_bgr_boxes_and_graph(esf_lib, name):
    """AVA.BGR true and false; FP64 / FP32 boxes on the host and on the device; K = 0; the default crop size
    (DATA.TEST_CROP_SIZE); a second call replays the same plan and graph; box count changes need no new plan."""
    for bgr in (False, True):
        cfg, model = _model(name, bgr=bgr)
        fr = _frames(cfg, 2, 240, 320, seed=7)
        boxes = _boxes(13, 2, seed=8)
        S = int(cfg.DATA.TEST_CROP_SIZE)
        xs, want_boxes = _oracle(cfg, model, fr, boxes, S, bgr)
        frd = fr.cuda()
        with torch.no_grad():
            want = model([t.cuda() for t in xs], want_boxes.cuda()).cpu()
            got = model.forward_ava_frames(frd, boxes)
            assert torch.equal(got.cpu(), want)
            plan = next(reversed(model._plans.values()))[1]
            graph = plan.graph
            for b in (boxes.cuda(), boxes.float(), boxes.float().cuda()):
                y, px = model.forward_ava_frames(frd, b, return_boxes=True)
                if b.dtype == torch.float64:
                    assert torch.equal(px.cpu(), want_boxes)
                else:      # FP32 boxes: the FP64 arithmetic of their FP32 values
                    _, wb = _oracle(cfg, model, fr, b.cpu(), S, bgr)
                    assert torch.equal(px.cpu(), wb)
                    assert torch.equal(y.cpu(), model([t.cuda() for t in xs], wb.cuda()).cpu())
            y, px = model.forward_ava_frames(frd, boxes.cuda(), return_boxes=True)
            assert torch.equal(y.cpu(), want) and torch.equal(px.cpu(), want_boxes)
            assert torch.equal(model.forward_ava_frames(frd, boxes[3:4]).cpu(), want[3:4])
            empty, eb = model.forward_ava_frames(frd, boxes[:0], return_boxes=True)
            assert empty.shape == (0, 80) and eb.shape == (0, 5) and empty.device.type == "cuda"
        assert len(model._plans) == 1 and next(iter(model._plans.values()))[1] is plan and plan.graph is graph
        assert graph is not None


def test_ava_frames_refusals_on_the_device(esf_lib):
    """The FP32 plan does not cover detection (NotImplementedError, as forward(x, bboxes)); host boxes with a batch
    index outside the batch raise ValueError before any launch."""
    cfg, model = _model("slow_r50", precision="fp32")
    fr = _frames(cfg, 1, 64, 96, seed=1).cuda()
    with pytest.raises(NotImplementedError):
        model.forward_ava_frames(fr, _boxes(2, 1, seed=2))
    cfg, model = _model("slow_r50")
    with pytest.raises(ValueError):
        model.forward_ava_frames(fr, torch.tensor([[1.0, 0.1, 0.1, 0.5, 0.5]]))
    assert len(model._plans) == 0
