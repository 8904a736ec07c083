"""Frames at capture size on the device: esf_resize_u8_cv2 equals cv2.resize(INTER_LINEAR) bit for bit on a ragged
sweep of sizes, writes nothing next to its outputs and nothing at all when an argument is bad; CameraWindows and
SlidingWindow with scale_to / bgr give, on every tick, what forward() gives on the demo's own inputs (cvtColor ->
cv2.resize -> demo_window_inputs) and what a plain bank gives on host-resized frames; detection boxes in capture
pixels equal host-scaled boxes (scale_boxes)."""
import ctypes

import numpy as np
import pytest
import torch

import helpers
from efficient_slowfast_b200 import CameraWindows, SlidingWindow
from efficient_slowfast_b200 import frames as F
from oracle import input_oracle as IO
from test_camera_capture import SIZES, TARGETS, cv2_scale, cv2_scale_boxes
from test_gpu_camera_windows import _ava_model

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

GUARD = 64          # sentinel bytes around every output


def test_resize_kernel_matches_cv2_on_a_ragged_sweep(esf_lib):
    """One call per C over every (size, target) of the sweep: 76 frames, two parameter chunks.  Every output equals
    cv2.resize; the guard bytes around every output keep their sentinel; a call with one bad frame at the end writes
    nothing."""
    rng = np.random.default_rng(0)
    for C in (1, 3, 4):
        srcs, jobs = [], []
        for H, W in SIZES:
            img = rng.integers(0, 256, (H, W, C), dtype=np.uint8)
            srcs.append((img, torch.from_numpy(img).cuda()))
            for S in TARGETS:
                jobs.append((len(srcs) - 1, F.Cv2Resize(H, W, S, "cuda")))
        assert len(jobs) > 64
        offsets, end = [], GUARD
        for _, r in jobs:
            offsets.append(end)
            end += r.Hs * r.Ws * C + GUARD
        out = torch.full((end,), 0xA5, dtype=torch.uint8, device="cuda")
        base = out.data_ptr()
        F.launch_resize_cv2([srcs[i][1].data_ptr() for i, _ in jobs], [base + o for o in offsets],
                            [r for _, r in jobs], C)
        host = out.cpu().numpy()
        guard = np.ones(end, bool)
        for (i, r), o in zip(jobs, offsets):
            n = r.Hs * r.Ws * C
            want = cv2.resize(srcs[i][0], (r.Ws, r.Hs), interpolation=cv2.INTER_LINEAR).reshape(-1)
            assert np.array_equal(host[o:o + n], want), (r.H, r.W, r.Hs, r.Ws, C)
            guard[o:o + n] = False
        assert np.all(host[guard] == 0xA5), C
        # the same call with a bad last frame: refused before any launch, nothing written
        fresh = torch.full((end,), 0xA5, dtype=torch.uint8, device="cuda")
        B = len(jobs)
        geom = [n for _, r in jobs for n in (r.H, r.W, r.Hs, r.Ws)]
        geom[-3] = 0
        rc = esf_lib.esf_resize_u8_cv2((ctypes.c_void_p * B)(*[srcs[i][1].data_ptr() for i, _ in jobs]),
                                       (ctypes.c_void_p * B)(*[fresh.data_ptr() + o for o in offsets]),
                                       (ctypes.c_int32 * (4 * B))(*geom),
                                       (ctypes.c_void_p * (2 * B))(*[a for _, r in jobs for a in (r.y.data_ptr(),
                                                                                                  r.x.data_ptr())]),
                                       B, C, None)
        assert rc < 0 and b"frame %d: bad size" % (B - 1) in esf_lib.esf_last_error()
        torch.cuda.synchronize()
        assert bool((fresh == 0xA5).all())


# cameras of three scaled sizes at S = 64: 64 x 85 (96 x 128 downscaled, 48 x 64 upscaled, 64 x 85 as it is),
# 64 x 113 (72 x 128) and portrait 85 x 64 (128 x 96)
CAMERAS = [(96, 128), (72, 128), (128, 96), (48, 64), (64, 85)]
JOIN = [0, 3, 7, 1, 5]
S = 64


def _model(name, precision="fp16", max_plans=3):
    cfg, model, _ = helpers.case_model_and_weights(name, precision)
    cfg.DATA.SAMPLING_RATE = 2
    cfg.ESF.MAX_PLANS = max_plans
    fam = model.__class__(cfg)
    fam.load_state_dict(model.state_dict())
    return cfg, fam.cuda().eval()


def _ticks(L, extra, join):
    full = max(join) + L - 1
    return [{c for c in range(len(join)) if k >= join[c] and not (c == 1 and k % 4 == 3 and k > full)}
            for k in range(full + 1 + extra)]


def _demo_frame(bgr):
    """What the demo appends to its buffer: cvtColor(BGR2RGB) then cv2_transform.scale to S."""
    return torch.from_numpy(np.ascontiguousarray(cv2_scale(S, cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB))))


def _window(cfg, model, history, L):
    alpha = None if model.num_pathways == 1 else int(cfg.SLOWFAST.ALPHA)
    return IO.demo_window_inputs(torch.stack(history[-L:]), cfg.DATA.MEAN, cfg.DATA.STD, int(cfg.DATA.NUM_FRAMES),
                                 alpha)


@pytest.mark.parametrize("name,precision", [("dual_r50", "fp16"), ("slow_r50", "fp16"), ("dual_r50", "fp32")])
def test_mixed_resolution_bank_equals_demo(esf_lib, name, precision):
    """CameraWindows(scale_to=64, bgr=True) over five cameras of four capture sizes and three scaled sizes, with
    staggered joins, a camera that skips pushes and one camera's frames on the device: every tick's scores equal
    forward() on the demo-assembled windows (each bank padded to its cameras, as the bank pads) and the rows of plain
    CameraWindows fed the host-resized RGB frames, bit for bit, in ascending camera id."""
    cfg, model = _model(name, precision)
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    bank = CameraWindows(model, cfg, len(CAMERAS), [h for h, _ in CAMERAS], [w for _, w in CAMERAS], scale_to=S,
                         bgr=True)
    assert [b.cameras for b in bank.banks] == [[0, 3, 4], [1], [2]]
    assert [b.frame_shape for b in bank.banks] == [(64, 85, 3), (64, 113, 3), (85, 64, 3)]
    plain = [CameraWindows(model, cfg, len(b.cameras), *b.frame_shape) for b in bank.banks]
    history = [[] for _ in CAMERAS]
    rng = np.random.default_rng(1)
    checked = 0
    for k, cams in enumerate(_ticks(L, 4, JOIN)):
        frames, plain_frames = {}, [{} for _ in plain]
        for c in sorted(cams):
            bgr = rng.integers(0, 256, CAMERAS[c] + (3,), dtype=np.uint8)
            frames[c] = torch.from_numpy(bgr).cuda() if c == 3 and k % 2 else torch.from_numpy(bgr).pin_memory()
            history[c].append(_demo_frame(bgr))
            g = bank._bank_of[c]
            plain_frames[bank.banks.index(g)][g.ring[c]] = history[c][-1].pin_memory()
        with torch.no_grad():
            res = bank.push(frames)
            plain_res = [p.push(f) for p, f in zip(plain, plain_frames)]
            ready = [c for c in sorted(cams) if len(history[c]) >= L]
            if res is None:
                assert not ready and all(r is None for r in plain_res)
                continue
            ids, scores = res
            assert ids == ready and scores.shape[0] == len(ids)
            want = {}
            for g, pr in zip(bank.banks, plain_res):
                rows = [c for c in ids if c in g.ring]
                if not rows:
                    assert pr is None
                    continue
                pad = rows + [rows[0]] * (len(g.cameras) - len(rows))
                per = [_window(cfg, model, history[c], L) for c in pad]
                ref = model([torch.cat([p[i] for p in per]).contiguous().cuda() for i in range(len(per[0]))])
                assert pr[0] == [g.ring[c] for c in rows]
                for r, c in enumerate(rows):
                    want[c] = ref[r]
                    assert torch.equal(pr[1][r], scores[ids.index(c)]), (k, c)
            assert torch.equal(scores, torch.stack([want[c] for c in ids])), (k, ids)
            checked += len(ids)
    assert checked >= 20
    print("%s %s: %d rows checked" % (name, precision, checked))


def test_sliding_window_at_capture_size(esf_lib):
    """SlidingWindow(scale_to=64, bgr=True) on 72 x 128 BGR captures equals a plain SlidingWindow fed the demo's
    resized RGB frames and forward() on the demo's window, bit for bit."""
    cfg, model = _model("dual_r50")
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    capture = SlidingWindow(model, cfg, 72, 128, scale_to=S, bgr=True)
    plain = SlidingWindow(model, cfg, 64, 113)
    rng = np.random.default_rng(2)
    history, checked = [], 0
    for k in range(L + 3):
        bgr = rng.integers(0, 256, (72, 128, 3), dtype=np.uint8)
        history.append(_demo_frame(bgr))
        with torch.no_grad():
            y = capture.push(torch.from_numpy(bgr).pin_memory())
            z = plain.push(history[-1].cuda())
            if k < L - 1:
                assert y is None and z is None
                continue
            want = model([t.contiguous().cuda() for t in _window(cfg, model, history, L)])
        assert torch.equal(y, z) and torch.equal(y, want), k
        checked += 1
    assert checked == 4


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_detection_boxes_in_capture_pixels(esf_lib, name):
    """An AVA model over cameras of two scaled sizes, boxes in capture pixels: the scores per camera equal plain banks
    fed the host-resized frames with the boxes scaled by cv2_transform.scale_boxes."""
    cfg, model = _ava_model(name)
    cams = [(96, 128), (72, 128), (96, 128)]
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    bank = CameraWindows(model, cfg, 3, [h for h, _ in cams], [w for _, w in cams], scale_to=S)
    plain = [CameraWindows(model, cfg, len(b.cameras), *b.frame_shape) for b in bank.banks]
    g = torch.Generator().manual_seed(7)
    rng = np.random.default_rng(3)
    checked = 0
    for k, ticking in enumerate(_ticks(L, 3, [0, 2, 4])):
        frames, boxes = {}, {}
        plain_frames, plain_boxes = [{} for _ in plain], [{} for _ in plain]
        for c in sorted(ticking):
            H, W = cams[c]
            rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
            frames[c] = torch.from_numpy(rgb)
            K = (k + c) % 3
            xy = torch.rand(K, 2, generator=g) * torch.tensor([W * 0.6, H * 0.6])
            wh = 4 + torch.rand(K, 2, generator=g) * torch.tensor([W * 0.4, H * 0.4])
            boxes[c] = torch.cat([xy, xy + wh], 1)
            b = bank._bank_of[c]
            i = bank.banks.index(b)
            plain_frames[i][b.ring[c]] = torch.from_numpy(np.ascontiguousarray(cv2_scale(S, rgb)))
            plain_boxes[i][b.ring[c]] = cv2_scale_boxes(S, boxes[c].clone(), H, W)
        with torch.no_grad():
            res = bank.push(frames, boxes)
            plain_res = [p.push(f, bx) for p, f, bx in zip(plain, plain_frames, plain_boxes)]
        if res is None:
            continue
        ids, scores = res
        for b, pr in zip(bank.banks, plain_res):
            if pr is None:
                continue
            for local, s in zip(*pr):
                c = b.cameras[local]
                assert torch.equal(scores[ids.index(c)], s), (k, c)
                checked += 1
    assert checked >= 8
