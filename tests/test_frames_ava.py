"""AVA detection from uint8 frames (forward_ava_frames), host side: the CPU restatement of the AVA test loader in
tests/ava_frames_oracle.py against the reference's functions, the resized sizes and axis tables against torch's own
bilinear weights, the kernel's arithmetic (resize of u / 255, then normalisation) emulated on the host, the box
arithmetic of esf_ava_boxes against the oracle, and argument validation.  No GPU needed."""
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import ava_frames_oracle as AO
from efficient_slowfast_b200 import config as C
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt
from oracle import ref_shim

# (H0, W0, S): AVA's 256 x 340 keyframes (a pure window at S = 256), 4:3, VGA, portrait, square, up- and down-scaling
GEOMETRIES = [(256, 340, 256), (240, 320, 256), (480, 640, 256), (340, 256, 256), (360, 202, 256), (300, 300, 256),
              (256, 340, 224), (97, 181, 112), (181, 97, 112), (255, 255, 128), (64, 96, 64), (48, 80, 64)]


def _onehot_weights(n_in, n_out):
    """torch's weights of one axis: dense [n_in][n_out] through one-hot rows of F.interpolate."""
    x = torch.zeros(1, n_in, n_in, 1)
    x[0, torch.arange(n_in), torch.arange(n_in), 0] = 1
    return F.interpolate(x, size=(n_out, 1), mode="bilinear", align_corners=False)[0, :, :, 0]


def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _emulate_ava(frames_u8, S, mean, std, chan_src):
    """What ava_frames_kernel computes for one clip (T, H, W, C): u / 255 looked up, blended with the axis tables in
    ATen's order (crop_value), then (v - mean[c]) / std[c] of the source channel, output channel c = source chan_src[c].
    Returns FP32 (C, T, Hr, Wr)."""
    T, H, W, Cn = frames_u8.shape
    Hr, Wr = FR.resized_size(H, W, S)
    lut = FR.unit_table(Cn).numpy()
    planes = np.stack([lut[c][frames_u8[..., c].numpy()] for c in range(Cn)])      # (C, T, H, W)
    if (Hr, Wr) != (H, W):
        yi, yw = (t.numpy() for t in FR.axis_table(H, Hr))
        xi, xw = (t.numpy() for t in FR.axis_table(W, Wr))
        r0, r1 = planes[:, :, yi[:, 0]], planes[:, :, yi[:, 1]]
        x00, x01, x10, x11 = r0[..., xi[:, 0]], r0[..., xi[:, 1]], r1[..., xi[:, 0]], r1[..., xi[:, 1]]
        w0, w1 = xw[:, 0], xw[:, 1]
        l0, l1 = yw[:, 0, None], yw[:, 1, None]
        t0 = _fma(x00, w0, (x01 * w1).astype(np.float32))
        t1 = _fma(x10, w0, (x11 * w1).astype(np.float32))
        planes = _fma(t0, l0, (t1 * l1).astype(np.float32))
    m = np.array(mean, dtype=np.float32)
    s = np.array(std, dtype=np.float32)
    out = [((planes[c] - m[c]) / s[c]).astype(np.float32) for c in range(Cn)]
    return torch.from_numpy(np.stack([out[c] for c in chan_src]))


@pytest.mark.parametrize("n_in,n_out", sorted({(h, r) for H0, W0, S in GEOMETRIES
                                               for h, r in zip((H0, W0), FR.resized_size(H0, W0, S))}))
def test_axis_tables_equal_torch_weights(n_in, n_out):
    idx, wt = FR.axis_table(n_in, n_out)
    want = torch.zeros(n_in, n_out)
    for d in range(n_out):
        i0, i1 = int(idx[d, 0]), int(idx[d, 1])
        if n_in == n_out:
            assert (i0, i1, float(wt[d, 0]), float(wt[d, 1])) == (d, 0, 1.0, 0.0)
            want[d, d] = 1
        elif i0 == i1:
            want[i0, d] = (wt[d, 0] + wt[d, 1]).item()
        else:
            assert i1 == i0 + 1
            want[i0, d], want[i1, d] = wt[d, 0], wt[d, 1]
    assert torch.equal(_onehot_weights(n_in, n_out), want)


@pytest.mark.parametrize("H0,W0,S", GEOMETRIES)
def test_resized_size_is_the_oracles(H0, W0, S):
    x = torch.zeros(1, 1, H0, W0)
    r, _ = AO.random_short_side_scale_jitter(x, S, boxes=np.zeros((0, 4)))
    assert FR.resized_size(H0, W0, S) == tuple(r.shape[2:])
    assert min(FR.resized_size(H0, W0, S)) == S


@pytest.mark.parametrize("bgr,reverse", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("H0,W0,S", [(48, 80, 64), (160, 120, 104), (64, 96, 64), (97, 181, 112), (121, 121, 104)])
def test_kernel_arithmetic_equals_oracle(H0, W0, S, bgr, reverse):
    """The kernel's value per element (emulated on the host) equals the loader chain bit for bit: the resize runs on
    u / 255 and the normalisation after it.  Resized widths of 104 or more and pure windows: below that width the CPU
    interpolate takes another contraction (DESIGN 3.7)."""
    g = torch.Generator().manual_seed(H0 * 1000 + W0)
    fr = torch.randint(0, 256, (1, 4, H0, W0, 3), generator=g, dtype=torch.uint8)
    mean, std = [0.45, 0.40, 0.35], [0.225, 0.25, 0.2]
    src = FR.ava_channel_source(3, bgr, reverse)
    want, _ = AO.prepare(fr, torch.zeros(0, 5), S, mean, std, 1, True, bgr, reverse)
    got = _emulate_ava(fr[0], S, mean, std, src)
    assert FR.resized_size(H0, W0, S)[1] >= 104 or FR.resized_size(H0, W0, S) == (H0, W0)
    assert torch.equal(got, want[0][0])


def _edge_boxes():
    """Boxes touching and crossing every edge, degenerate (zero area, x1 > x2), exactly on the corners, far outside,
    and interior ones; rows [batch index, x1, y1, x2, y2] in [0, 1] coordinates (and beyond)."""
    rows = [[0, 0.0, 0.0, 1.0, 1.0], [0, -0.2, -0.1, 1.3, 1.2], [0, 0.5, 0.5, 0.5, 0.5], [0, 0.7, 0.6, 0.2, 0.1],
            [0, 1.0, 1.0, 1.0, 1.0], [0, 0.0, 0.0, 0.0, 0.0], [0, -1.0, -1.0, -0.5, -0.5], [0, 1.5, 1.5, 2.0, 2.0],
            [0, 0.999, 0.001, 1.0, 0.002], [0, 0.25, 0.1, 0.75, 0.9], [0, 0.1, 0.995, 0.9, 1.0],
            [0, 1 / 3, 2 / 3, 0.7521, 0.99999]]
    g = torch.Generator().manual_seed(4)
    rnd = torch.rand(40, 4, generator=g, dtype=torch.float64) * 1.4 - 0.2
    return torch.cat([torch.tensor(rows, dtype=torch.float64),
                      torch.cat([torch.zeros(40, 1, dtype=torch.float64), rnd], 1)])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("H0,W0,S", GEOMETRIES)
def test_box_arithmetic_equals_oracle(H0, W0, S, dtype):
    boxes = _edge_boxes().to(dtype)
    fr = torch.zeros(1, 1, H0, W0, 3, dtype=torch.uint8)
    _, want = AO.prepare(fr, boxes, S, [0.0] * 3, [1.0] * 3, 1, True)
    got = FR.ava_boxes(boxes.numpy(), H0, W0, S)
    assert got.dtype == torch.float32 and torch.equal(got, want)
    # the final clip is to S x S, also along the long side (the reference's test branch keeps its quirk)
    assert float(got[:, 1:].max()) <= S - 1


def test_box_rows_keep_their_clip():
    """Boxes of several clips in any order: each row is transformed with its own clip's geometry (one geometry per
    batch here) and keeps its position and batch index."""
    boxes = torch.tensor([[1, 0.1, 0.2, 0.3, 0.4], [0, 0.5, 0.5, 0.9, 0.9], [1, 0.0, 0.0, 1.0, 1.0]], dtype=torch.float64)
    fr = torch.zeros(2, 1, 240, 320, 3, dtype=torch.uint8)
    _, want = AO.prepare(fr, boxes, 256, [0.0] * 3, [1.0] * 3, 1, True)
    assert torch.equal(FR.ava_boxes(boxes.numpy(), 240, 320, 256), want)
    assert want[:, 0].tolist() == [1.0, 0.0, 1.0]


def test_channel_source():
    assert FR.ava_channel_source(3) == [2, 1, 0]                      # AVA.BGR false: BGR -> RGB
    assert FR.ava_channel_source(3, bgr=True) == [0, 1, 2]
    assert FR.ava_channel_source(3, reverse=True) == [0, 1, 2]        # swapped twice
    assert FR.ava_channel_source(3, bgr=True, reverse=True) == [2, 1, 0]
    assert FR.ava_channel_source(1, bgr=True) == [0]
    with pytest.raises(ValueError):
        FR.ava_channel_source(1)


def test_unit_table_is_the_loaders_division():
    u = torch.arange(256, dtype=torch.uint8)
    t = FR.unit_table(3)
    assert t.shape == (3, 256) and t.dtype == torch.float32
    for c in range(3):
        assert torch.equal(t[c], u.float() / 255.0)


@pytest.fixture(scope="module")
def ava_slow():
    from efficient_slowfast_b200 import build_model

    cfg = C.ava_slow_8x8_r50_cfg()
    cfg.NUM_GPUS = 0
    torch.manual_seed(0)
    return build_model(cfg).eval()


def test_validation_raises_before_anything_runs(ava_slow, monkeypatch):
    """Bad arguments raise ValueError (NotImplementedError for what is not covered) before any plan is compiled or
    kernel launched: the library is not even loaded."""
    model = ava_slow

    def no_lib():
        raise AssertionError("the library was reached")

    monkeypatch.setattr(rt, "lib", no_lib)
    fr = torch.zeros(2, 8, 64, 96, 3, dtype=torch.uint8)
    ok = torch.tensor([[0, 0.1, 0.1, 0.5, 0.5], [1, 0.2, 0.2, 0.9, 0.9]])
    for bad in (fr.float(), fr[..., 0], fr.permute(0, 1, 3, 2, 4), [fr], torch.zeros(2, 8, 8, 5000, 4, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            model.forward_ava_frames(bad, ok)
    for bad in (None, ok[:, :4], ok.long(), ok[None], torch.tensor([[2.0, 0, 0, 1, 1]]),
                torch.tensor([[-1.0, 0, 0, 1, 1]]), torch.tensor([[float("nan"), 0, 0, 1, 1]])):
        with pytest.raises(ValueError):
            model.forward_ava_frames(fr, bad)
    with pytest.raises(ValueError):
        model.forward_ava_frames(fr, ok, crop_size=0)
    with pytest.raises(rt.EsfError):
        model.forward_ava_frames(fr, ok)                                # valid arguments: refused only for the device
    model.train()
    with pytest.raises(NotImplementedError):
        model.forward_ava_frames(fr, ok)
    model.eval()


def test_not_covered_raises_not_implemented(monkeypatch):
    from efficient_slowfast_b200 import build_model

    monkeypatch.setattr(rt, "lib", lambda: (_ for _ in ()).throw(AssertionError("the library was reached")))
    fr = torch.zeros(1, 8, 64, 96, 3, dtype=torch.uint8)
    ok = torch.tensor([[0, 0.1, 0.1, 0.5, 0.5]])
    cfg = C.resnet_cfg("slow", num_frames=8)                          # a classification model
    cfg.NUM_GPUS = 0
    torch.manual_seed(0)
    with pytest.raises(NotImplementedError):
        build_model(cfg).eval().forward_ava_frames(fr, ok)
    cfg = C.ava_slow_8x8_r50_cfg()
    cfg.NUM_GPUS = 0
    cfg.AVA = cfg.DATA.__class__(dict(TEST_FORCE_FLIP=True))
    with pytest.raises(NotImplementedError):
        build_model(cfg).eval().forward_ava_frames(fr, ok)


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not mounted (ESF_REFERENCE_ROOT)")
def test_oracle_matches_reference_transforms():
    ref_shim.reference_dataset_utils()
    Tr = importlib.import_module("slowfast.datasets.transform")
    g = torch.Generator().manual_seed(8)
    boxes = _edge_boxes()[:, 1:].numpy()
    for H0, W0, S in GEOMETRIES[:8]:
        x = torch.rand(3, 3, H0, W0, generator=g)
        b = AO.clip_boxes_to_image(boxes * [W0, H0, W0, H0], H0, W0)
        assert np.array_equal(b, Tr.clip_boxes_to_image(boxes * [W0, H0, W0, H0], H0, W0))
        r, rb = Tr.random_short_side_scale_jitter(x, S, S, boxes=b)
        o, ob = AO.random_short_side_scale_jitter(x, S, boxes=b)
        assert torch.equal(o, r) and np.array_equal(ob, rb)
        m, s = np.array([0.45, 0.4, 0.35], dtype=np.float32), np.array([0.225, 0.25, 0.2], dtype=np.float32)
        assert torch.equal(AO.color_normalization(o, m, s), Tr.color_normalization(r, m, s))
