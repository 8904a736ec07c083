"""Frames at capture size for the demo loop (no GPU): the per-axis tables of frames.cv2_axis_table restate OpenCV's
uint8 cv2.resize(INTER_LINEAR) bit for bit, the size rule and box scaling are those of the reference's
datasets/cv2_transform.scale / scale_boxes, and CameraWindows(scale_to=...) refuses what it cannot run before it
allocates anything."""
import math

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

# capture sizes (H, W): common camera modes, portrait, odd sizes, upscales, exact 2x downscales and frames whose short
# side already is the target
SIZES = [(1080, 1920), (720, 1280), (480, 640), (2160, 3840), (1920, 1080), (57, 91), (91, 57), (1001, 1000),
         (1000, 1001), (100, 100), (448, 796), (448, 448), (224, 398), (240, 320), (256, 340), (96, 128), (128, 96),
         (48, 64), (64, 85)]
TARGETS = (112, 160, 224, 256)


def cv2_resize_restated(img, Hs, Ws):
    """cv2.resize(img, (Ws, Hs), INTER_LINEAR) on uint8 (H, W, C) from the tables of cv2_axis_table, integers only."""
    from efficient_slowfast_b200.frames import cv2_axis_table

    H, W, _ = img.shape
    yt, xt = cv2_axis_table(H, Hs, False), cv2_axis_table(W, Ws, True)
    p = img.astype(np.int64)
    x0, x1 = np.clip(xt["index"], 0, W - 1), np.clip(xt["index"] + 1, 0, W - 1)
    rows = p[:, x0] * xt["w0"].astype(np.int64)[:, None] + p[:, x1] * xt["w1"].astype(np.int64)[:, None]
    y0, y1 = np.clip(yt["index"], 0, H - 1), np.clip(yt["index"] + 1, 0, H - 1)
    b0, b1 = yt["w0"].astype(np.int64)[:, None, None], yt["w1"].astype(np.int64)[:, None, None]
    v = (((b0 * (rows[y0] >> 4)) >> 16) + ((b1 * (rows[y1] >> 4)) >> 16) + 2) >> 2
    return np.clip(v, 0, 255).astype(np.uint8)


def cv2_scale(size, image):
    """datasets/cv2_transform.scale, with the returned frame kept as uint8 (the reference casts it to float32; the
    values are the same integers)."""
    height, width = image.shape[0], image.shape[1]
    if (width <= height and width == size) or (height <= width and height == size):
        return image
    new_width = new_height = size
    if width < height:
        new_height = int(math.floor((float(height) / width) * size))
    else:
        new_width = int(math.floor((float(width) / height) * size))
    out = cv2.resize(image, (new_width, new_height), interpolation=cv2.INTER_LINEAR)
    return out.reshape(out.shape[0], out.shape[1], -1)


def cv2_scale_boxes(size, boxes, height, width):
    """datasets/cv2_transform.scale_boxes (in place on the FP32 torch boxes)."""
    if (width <= height and width == size) or (height <= width and height == size):
        return boxes
    if width < height:
        new_height = int(math.floor((float(height) / width) * size))
        boxes *= float(new_height) / height
    else:
        new_width = int(math.floor((float(width) / height) * size))
        boxes *= float(new_width) / width
    return boxes


def test_axis_tables_restate_cv2_resize():
    """The integer restatement equals cv2.resize over the sweep for C = 1, 3, 4.  C = 2 is refused by the kernel and
    CameraWindows: at an exact 2x downscale OpenCV switches to INTER_AREA, and there the restatement differs."""
    from efficient_slowfast_b200.frames import resized_size

    rng = np.random.default_rng(0)
    checked = 0
    for H, W in SIZES:
        for S in TARGETS:
            Hs, Ws = resized_size(H, W, S)
            for C in (1, 3, 4):
                img = rng.integers(0, 256, (H, W, C), dtype=np.uint8)
                want = cv2.resize(img, (Ws, Hs), interpolation=cv2.INTER_LINEAR).reshape(Hs, Ws, C)
                assert np.array_equal(cv2_resize_restated(img, Hs, Ws), want), (H, W, S, C)
                checked += 1
    assert checked == len(SIZES) * len(TARGETS) * 3
    img = rng.integers(0, 256, (448, 796, 2), dtype=np.uint8)                 # exact 2x: INTER_AREA in OpenCV
    want = cv2.resize(img, (398, 224), interpolation=cv2.INTER_LINEAR)
    assert not np.array_equal(cv2_resize_restated(img, 224, 398), want)


def test_axis_table_layout_and_edges():
    from efficient_slowfast_b200.frames import CV2_AXIS, cv2_axis_table

    assert CV2_AXIS.itemsize == 8
    up_x, up_y = cv2_axis_table(100, 224, True), cv2_axis_table(100, 224, False)
    assert up_x["index"][0] == 0 and up_x["w1"][0] == 0                        # clamped: s < 0 -> (0, f = 0)
    assert up_y["index"][0] == -1 and up_y["w1"][0] > 0                        # the y axis keeps s and f
    assert up_x["index"][-1] == 99 and up_x["w1"][-1] == 0
    assert np.all(up_x["w0"].astype(int) + up_x["w1"] == 2048)
    same = cv2_axis_table(224, 224, True)
    assert np.array_equal(same["index"], np.arange(224)) and np.all(same["w0"] == 2048)


def test_size_rule_and_boxes_match_cv2_transform():
    from efficient_slowfast_b200.frames import resized_size, scale_boxes

    rng = np.random.default_rng(1)
    for H, W in SIZES:
        for S in TARGETS:
            img = np.zeros((H, W, 1), np.uint8)
            assert cv2_scale(S, img).shape[:2] == resized_size(H, W, S), (H, W, S)
            boxes = torch.from_numpy(rng.uniform(0, max(H, W), (5, 4)).astype(np.float32))
            want = cv2_scale_boxes(S, boxes.clone(), H, W)
            got = scale_boxes(S, boxes, H, W)
            assert got.dtype == torch.float32 and torch.equal(got, want), (H, W, S)
    b = torch.ones(1, 4, dtype=torch.float32)
    scale_boxes(112, b, 480, 640)
    assert torch.equal(b, torch.ones(1, 4))                                    # the caller's boxes stay as they are


class _Model(torch.nn.Module):
    """What CameraWindows reads of a model before it touches a device."""
    num_pathways = 1

    def __init__(self, max_plans=2, max_batch=0):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1, device="meta"))
        self._max_plans, self._max_batch = max_plans, max_batch


def _cfg():
    from efficient_slowfast_b200 import config

    cfg = config.get_cfg()
    cfg.DATA.NUM_FRAMES, cfg.DATA.SAMPLING_RATE = 4, 2
    return cfg


def test_constructor_refusals():
    """ValueError for every layout CameraWindows(scale_to=...) cannot run, before it allocates (the model's parameters
    are on the meta device: a check that came after the device check would raise EsfError instead)."""
    from efficient_slowfast_b200 import CameraWindows

    cfg = _cfg()
    cases = [
        dict(model=_Model(max_plans=2), cameras=3, height=[96, 72, 128], width=[128, 128, 96], scale_to=64),  # 3 sizes
        dict(model=_Model(), cameras=2, height=480, width=640, channels=2, scale_to=224),                     # C = 2
        dict(model=_Model(), cameras=3, height=[480, 720], width=640, scale_to=224),                          # 2 of 3
        dict(model=_Model(), cameras=2, height=[480, 720, 1080], width=[640] * 3, scale_to=224),              # 3 of 2
        dict(model=_Model(), cameras=2, height=[480, 0], width=[640, 640], scale_to=224),                     # size 0
        dict(model=_Model(), cameras=2, height=[480, 480], width=[640, 640]),                                 # no scale_to
        dict(model=_Model(), cameras=2, height=480, width=640, scale_to=0),
        dict(model=_Model(), cameras=2, height=480, width=640, channels=4, scale_to=224, bgr=True),            # bgr, C 4
        dict(model=_Model(), cameras=1, height=480, width=8192, scale_to=224),                                # row bytes
        dict(model=_Model(max_batch=1), cameras=2, height=480, width=640, scale_to=224),                      # MAX_BATCH
    ]
    for kw in cases:
        model = kw.pop("model")
        with pytest.raises(ValueError):
            CameraWindows(model, cfg, **kw)


def test_check_push_with_per_camera_shapes():
    from efficient_slowfast_b200 import demo

    clock = demo.CameraClock(3, 2, 1)
    shapes = [(6, 8, 3), (8, 6, 3), (6, 8, 3)]
    f = {c: torch.zeros(s, dtype=torch.uint8) for c, s in enumerate(shapes)}
    ids, ready, b, counts = demo.check_push(dict(f), None, clock, shapes, torch.device("cuda", 0), False)
    assert ids == [0, 1, 2] and ready == [] and b is None and counts is None
    for bad in ({1: f[0]}, {0: f[1]}, {2: torch.zeros((6, 8, 4), dtype=torch.uint8)}):
        with pytest.raises(ValueError):
            demo.check_push(bad, None, clock, shapes, torch.device("cuda", 0), False)
    clock.advance([0, 1, 2])
    boxes = {0: torch.tensor([[1.0, 2.0, 3.0, 4.0]]), 1: torch.zeros((0, 4))}
    ids, ready, rows, counts = demo.check_push({0: f[0], 1: f[1]}, boxes, clock, shapes, torch.device("cuda", 0), True)
    assert ready == [0, 1] and counts == [1, 0] and torch.equal(rows, torch.tensor([[0.0, 1.0, 2.0, 3.0, 4.0]]))
    assert clock.count == [1, 1, 1]


def test_library_refuses_bad_resize_arguments(esf_lib):
    """esf_resize_u8_cv2 checks every frame before it launches: each call below has a null or unaligned address or a
    bad size somewhere and returns an error without reaching a launch."""
    import ctypes

    fake = 256                                   # never dereferenced: every call is refused on the host

    def call(geom, C=3, B=None, src=fake, dst=fake, tab=fake):
        B = len(geom) // 4 if B is None else B
        n = max(B, 1)
        return (esf_lib.esf_resize_u8_cv2((ctypes.c_void_p * n)(*[src] * n), (ctypes.c_void_p * n)(*[dst] * n),
                                          (ctypes.c_int32 * len(geom))(*geom),
                                          (ctypes.c_void_p * (2 * n))(*[tab] * (2 * n)), B, C, None),
                esf_lib.esf_last_error())

    cases = [
        (dict(geom=[480, 640, 224, 298], B=0), b"null/bad argument"),
        (dict(geom=[480, 640, 224, 298], C=2), b"2 channels"),
        (dict(geom=[480, 640, 224, 298], C=5), b"5 channels"),
        (dict(geom=[480, 640, 224, 298], src=0), b"frame 0: null address"),
        (dict(geom=[480, 640, 224, 298], dst=0), b"frame 0: null address"),
        (dict(geom=[480, 640, 224, 298], tab=260), b"misaligned axis table"),
        (dict(geom=[480, 640, 224, 298, 480, 0, 224, 298]), b"frame 1: bad size"),
        (dict(geom=[480, 8192, 224, 298]), b"exceed 16384"),
    ]
    for kw, msg in cases:
        rc, err = call(**kw)
        assert rc < 0 and msg in err and b"launch" not in err, (kw, rc, err)
