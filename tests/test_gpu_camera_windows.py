"""demo.CameraWindows on the device: every tick's rows equal forward() on the inputs the reference demo would assemble on
the host for the same cameras' windows, stacked in the same order, bit for bit; each row agrees with a single-camera
SlidingWindow fed the same frames; the batch-capacity route keeps one plan family and replays graphs; the padded route
(no MAX_BATCH) and an AVA detection model with per-camera boxes."""
import pytest
import torch

import helpers
from efficient_slowfast_b200 import CameraWindows, SlidingWindow
from efficient_slowfast_b200.workloads import seeded_state_dict
from oracle import input_oracle as IO

pytestmark = pytest.mark.gpu

N = 3
JOIN = [0, 3, 7]                  # tick at which each camera starts to push
SIZES = [(64, 64), (64, 340)]     # the packed 16-bit stem rows, and the FP32 clip of the CUDA-core stem fallback


def _model(name, precision="fp16", max_batch=0):
    cfg, model, _ = helpers.case_model_and_weights(name, precision)
    cfg.DATA.SAMPLING_RATE = 2
    if max_batch:
        cfg.ESF.MAX_BATCH = max_batch
        fam = model.__class__(cfg)
        fam.load_state_dict(model.state_dict())
        model = fam
    return cfg, model.cuda().eval()


def _ticks(L, extra):
    """Cameras pushing on every tick: staggered joins; once every window can be full, camera 1 skips every fourth tick."""
    full = JOIN[-1] + L - 1
    return [{c for c in range(N) if k >= JOIN[c] and not (c == 1 and k % 4 == 3 and k > full)}
            for k in range(full + 1 + extra)]


def _alpha(cfg, model):
    return None if model.num_pathways == 1 else int(cfg.SLOWFAST.ALPHA)


def _stacked(cfg, model, history, cams, L):
    nf = int(cfg.DATA.NUM_FRAMES)
    per = [IO.demo_window_inputs(torch.stack(history[c][-L:]), cfg.DATA.MEAN, cfg.DATA.STD, nf, _alpha(cfg, model))
           for c in cams]
    return [torch.cat([p[i] for p in per]).contiguous().cuda() for i in range(len(per[0]))]


def _run(cfg, model, H, W, stride=1, seed=0, hooks=None):
    """Drive a CameraWindows and N SlidingWindows with the same frames; check every tick against forward() on the
    stacked host-assembled inputs (padded with row 0 when the bank pads).  Returns (ticks with rows, rows checked,
    rows bit-identical to the SlidingWindow's, set of R seen, packed-route flags of the plans used)."""
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    bank = CameraWindows(model, cfg, N, H, W, stride=stride)
    singles = [SlidingWindow(model, cfg, H, W) for _ in range(N)]
    history = [[] for _ in range(N)]
    g = torch.Generator().manual_seed(seed)
    ticks = rows = identical = 0
    seen, routes = set(), set()
    for k, cams in enumerate(_ticks(L, 3 * stride + 3)):
        frames = {}
        for c in sorted(cams):
            frames[c] = torch.randint(0, 256, (H, W, 3), generator=g, dtype=torch.uint8).pin_memory()
            history[c].append(frames[c])
        with torch.no_grad():
            res = bank.push(frames)
            if res is not None:
                plan = next(reversed(model._plans.values()))[1]       # the bank's plan (family) is the latest used
                plan = plan.variants.get(len(res[0]), plan) if model._max_batch else plan
                routes.add(tuple(own.data_ptr() in plan.stem_routes for own in plan.inputs))
            single = {c: singles[c].push(frames[c]) for c in sorted(cams)}
            if res is None:
                assert all(y is None or (len(history[c]) - L) % stride for c, y in single.items())
                continue
            ids, scores = res
            R = len(ids)
            assert ids == sorted(ids) and scores.shape == (R, int(cfg.MODEL.NUM_CLASSES))
            assert ids == [c for c in sorted(cams) if len(history[c]) >= L and (len(history[c]) - L) % stride == 0]
            pad = ids + [ids[0]] * ((N if bank.padded else R) - R)
            want = model(_stacked(cfg, model, history, pad, L))[:R]
            assert torch.equal(scores, want), (k, ids)
            for r, c in enumerate(ids):
                y = single[c]
                assert y is not None and torch.equal(y.argmax(1), scores[r:r + 1].argmax(1)), (k, c)
                assert helpers.rel_err(scores[r:r + 1].cpu(), y.cpu()) <= 2e-2, (k, c)
                identical += int(torch.equal(y, scores[r:r + 1]))
            ticks, rows = ticks + 1, rows + R
            seen.add(R)
            if hooks:
                hooks(k, R)
    return ticks, rows, identical, seen, routes


@pytest.mark.parametrize("name,precision", [("dual_r50", "fp16"), ("slow_r50", "fp16"), ("dual_r50", "fp32"),
                                            ("slow_r50", "fp32")])
def test_camera_windows_with_batch_capacity(esf_lib, monkeypatch, name, precision):
    """MAX_BATCH = cameras: every tick is bit-identical to forward() on the stacked demo inputs; one LRU entry serves
    every R, nothing compiles after the first tick of each R, and later ticks replay the captured graphs."""
    cfg, model = _model(name, precision, max_batch=N)
    compiled, replays = [], [0]
    compile_plan = model._compile_plan
    monkeypatch.setattr(model, "_compile_plan", lambda shapes, *a, **k: compiled.append(shapes[0][0]) or
                        compile_plan(shapes, *a, **k))
    replay = torch.cuda.CUDAGraph.replay
    monkeypatch.setattr(torch.cuda.CUDAGraph, "replay", lambda self: replays.__setitem__(0, replays[0] + 1) or replay(self))
    routes = set()
    for i, (H, W) in enumerate(SIZES):
        seen_r, count = set(), [len(compiled)]

        def hooks(k, R):
            new, count[0] = len(compiled) - count[0], len(compiled)
            assert R not in seen_r or new == 0, "tick %d compiled %d plans for R = %d, seen before" % (k, new, R)
            seen_r.add(R)

        before = replays[0]
        ticks, rows, identical, seen, used = _run(cfg, model, H, W, seed=i, hooks=hooks)
        routes |= used
        assert seen == {1, 2, 3} and ticks >= 8
        assert len(model._plans) == i + 1                 # one family for every R of a frame size
        cap = next(reversed(model._plans.values()))[1]
        assert sorted(cap.variants) == [1, 2] and all(p.graph is not None for p in [cap] + list(cap.variants.values()))
        assert replays[0] - before >= 2 * ticks           # the bank's forward and the reference forward of every tick
        print("%s %s %dx%d: %d ticks, %d rows, %d bit-identical to SlidingWindow, stem routes %s"
              % (name, precision, H, W, ticks, rows, identical, sorted(used)))
    if precision == "fp32":      # the FP32-accurate plan packs its stem from the FP32 clip (hi / lo halves) at every size
        assert routes == {(False,) * model.num_pathways}, routes
    else:
        assert len({r for rs in routes for r in rs}) == 2, "the frame sizes must cover both stem routes: %s" % routes


@pytest.mark.parametrize("name", ["dual_r50", "slow_r50"])
def test_camera_windows_padded_without_batch_capacity(esf_lib, name):
    """MAX_BATCH off: every tick runs the plan of `cameras` rows (padding rows repeat row 0) and the rows equal
    forward() on the same padded stack; stride 2 predicts on every other frame of each camera."""
    cfg, model = _model(name)
    for i, (H, W) in enumerate(SIZES):
        ticks, rows, identical, seen, _ = _run(cfg, model, H, W, stride=2, seed=10 + i)
        assert {1, 2} & seen and ticks >= 4
        print("%s padded %dx%d: %d ticks, %d rows, %d bit-identical to SlidingWindow" % (name, H, W, ticks, rows,
                                                                                        identical))


def _ava_model(name):
    cfg = helpers.case_cfg(name)
    npw = len(cfg.DATA.INPUT_CHANNEL_NUM)
    cfg.RESNET.SPATIAL_STRIDES = [[1] * npw, [2] * npw, [2] * npw, [1] * npw]
    cfg.RESNET.SPATIAL_DILATIONS = [[1] * npw, [1] * npw, [1] * npw, [2] * npw]
    cfg.DETECTION.ENABLE = True
    cfg.MODEL.NUM_CLASSES, cfg.MODEL.HEAD_ACT = 80, "sigmoid"
    cfg.MULTIGRID.SHORT_CYCLE = False
    cfg.DATA.SAMPLING_RATE = 2
    from efficient_slowfast_b200 import build_model

    torch.manual_seed(0)
    model = build_model(cfg)
    gold = helpers.load_golden(name)
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    model.load_state_dict(seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    return cfg, model.eval().cuda()


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_camera_windows_detection_boxes(esf_lib, name):
    """AVA detection: per-camera pixel boxes become (K, 5) rows with batch index = row; the scores, split per camera,
    equal forward(stacked demo inputs, boxes); a ready camera without boxes is refused before anything runs."""
    cfg, model = _ava_model(name)
    H, W = 64, 96
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    bank = CameraWindows(model, cfg, N, H, W)
    history = [[] for _ in range(N)]
    g = torch.Generator().manual_seed(5)
    checked = 0
    for k, cams in enumerate(_ticks(L, 3)):
        frames, boxes = {}, {}
        for c in sorted(cams):
            frames[c] = torch.randint(0, 256, (H, W, 3), generator=g, dtype=torch.uint8)
            K = 1 + (k + c) % 3
            xy = torch.rand(K, 2, generator=g) * torch.tensor([W * 0.6, H * 0.6])
            wh = 4 + torch.rand(K, 2, generator=g) * torch.tensor([W * 0.4, H * 0.4])
            boxes[c] = torch.cat([xy, xy + wh], 1)
            if c == 2 and k % 2:
                boxes[c] = boxes[c].cuda()
        ready = [c for c in sorted(cams) if len(history[c]) + 1 >= L]
        if ready:
            counts = list(bank.clock.count)
            with pytest.raises(ValueError):
                bank.push(frames, {c: b for c, b in boxes.items() if c != ready[0]})
            assert bank.clock.count == counts
        for c in sorted(cams):
            history[c].append(frames[c])
        with torch.no_grad():
            res = bank.push(frames, boxes)
            if res is None:
                continue
            ids, scores = res
            assert ids == ready and len(scores) == len(ids)
            rows = torch.cat([torch.cat([torch.full((boxes[c].shape[0], 1), float(r)), boxes[c].cpu()], 1)
                              for r, c in enumerate(ids)])
            pad = ids + [ids[0]] * (N - len(ids))
            want = model(_stacked(cfg, model, history, pad, L), rows)
            assert torch.equal(torch.cat(scores), want), (k, ids)
            assert [s.shape[0] for s in scores] == [boxes[c].shape[0] for c in ids]
            checked += len(ids)
    assert checked >= 8
