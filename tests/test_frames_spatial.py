"""Test-time spatial sampling of uint8 frames (forward_frames(crop_size=, spatial_idx=)), host side: the CPU restatement
in tests/spatial_oracle.py against the reference's functions, the per-axis resize tables of frames.axis_table against
torch's own bilinear weights, crop offsets, row order and argument validation.  No GPU needed."""
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import helpers
import spatial_oracle as SO
from efficient_slowfast_b200 import frames as FR
from oracle import input_oracle as IO
from oracle import ref_shim

# (H0, W0, S): landscape / portrait / square, odd sizes, sizes already at the short side, up- and down-scaling
GEOMETRIES = [(256, 340, 224), (340, 256, 224), (240, 320, 224), (720, 1280, 256), (224, 298, 224), (224, 224, 224),
              (256, 340, 256), (181, 97, 112), (97, 181, 112), (100, 100, 112), (128, 171, 224), (1080, 1920, 256),
              (255, 255, 128), (33, 517, 32)]


def _onehot_weights(n_in, n_out):
    """torch's weights of one axis: dense [n_in][n_out], column d holds what interpolate gives every source row for
    output row d (one-hot rows through F.interpolate, the other axis of size 1 -> 1 is the identity)."""
    x = torch.zeros(1, n_in, n_in, 1)
    x[0, torch.arange(n_in), torch.arange(n_in), 0] = 1
    return F.interpolate(x, size=(n_out, 1), mode="bilinear", align_corners=False)[0, :, :, 0]


def _fma(a, b, c):
    """FP32 fused multiply-add (the FP64 product of two FP32 numbers is exact; one rounding of the sum)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _emulate_resize(planes, yi, yw, xi, xw):
    """What crop_frames_kernel computes per (plane, row, column) from the tables (csrc/esf_crop.cu crop_value)."""
    yi, yw, xi, xw = (t.numpy() for t in (yi, yw, xi, xw))
    r0, r1 = planes[:, yi[:, 0]], planes[:, yi[:, 1]]
    x00, x01, x10, x11 = r0[:, :, xi[:, 0]], r0[:, :, xi[:, 1]], r1[:, :, xi[:, 0]], r1[:, :, xi[:, 1]]
    w0, w1 = xw[None, None, :, 0], xw[None, None, :, 1]
    l0, l1 = yw[None, :, None, 0], yw[None, :, None, 1]
    t0 = _fma(x00, w0, (x01 * w1).astype(np.float32))
    t1 = _fma(x10, w0, (x11 * w1).astype(np.float32))
    return _fma(t0, l0, (t1 * l1).astype(np.float32))


@pytest.mark.parametrize("n_in,n_out", sorted({(h, r) for H0, W0, S in GEOMETRIES
                                               for h, r in zip((H0, W0), FR.resized_size(H0, W0, S))}))
def test_axis_table_equals_torch_weights(n_in, n_out):
    """Every (index, weight) pair of the table is what torch's CPU interpolate uses, exactly.  Where both taps read the
    same source row (the clamped border of an upscale) torch can only show their sum, and that sum must match."""
    idx, wt = FR.axis_table(n_in, n_out)
    assert idx.dtype == torch.int32 and wt.dtype == torch.float32 and tuple(idx.shape) == (n_out, 2)
    assert int(idx.min()) >= 0 and int(idx.max()) < n_in
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
def test_tables_reproduce_torch_interpolate(H0, W0, S):
    """The kernel's blend (ATen's order and FMA use) over the tables == F.interpolate on the reference's (C, T, H, W)
    layout, bit for bit, on N(0, 1) values.  (Every resized width here is >= 104: torch's CPU kernel contracts the
    blend differently for narrower outputs, see DESIGN 3.7.)"""
    Hr, Wr = FR.resized_size(H0, W0, S)
    g = torch.Generator().manual_seed(H0 * 7 + W0)
    x = torch.randn(2, H0, W0, 3, generator=g).permute(3, 0, 1, 2)          # (C, T, H, W) view, like the loader's
    ref = SO.random_short_side_scale_jitter(x, S)
    assert tuple(ref.shape[2:]) == (Hr, Wr)
    yi, yw = FR.axis_table(H0, Hr)
    xi, xw = FR.axis_table(W0, Wr)
    got = _emulate_resize(x.reshape(-1, H0, W0).contiguous().numpy(), yi, yw, xi, xw).reshape(ref.shape)
    assert np.array_equal(got, ref.numpy())


@pytest.mark.parametrize("H0,W0,S", GEOMETRIES)
def test_crop_offsets_match_uniform_crop(H0, W0, S):
    """frames.crop_offset == the window uniform_crop cuts, for the three indices, both orientations."""
    Hr, Wr = FR.resized_size(H0, W0, S)
    grid = torch.arange(Hr * Wr, dtype=torch.float64).reshape(1, 1, Hr, Wr)
    for idx in (0, 1, 2):
        y0, x0 = FR.crop_offset(Hr, Wr, S, idx)
        c = SO.uniform_crop(grid, S, idx)
        assert tuple(c.shape[2:]) == (S, S)
        assert int(c[0, 0, 0, 0]) == y0 * Wr + x0
    if Hr > Wr:
        assert [FR.crop_offset(Hr, Wr, S, i)[0] for i in (0, 2)] == [0, Hr - S]
    elif Wr > Hr:
        assert [FR.crop_offset(Hr, Wr, S, i)[1] for i in (0, 2)] == [0, Wr - S]


def _emulate_crop_route(fin, frames, size, views, t_out, alpha):
    """crop_frames_kernel on the CPU: lut32 gather of the source channel, resize from the tables, crop, frame gather;
    rows b * V + v."""
    B, T, H0, W0, C = frames.shape
    tabs = fin.crop(H0, W0, size, views)
    idx = fin.index(T, t_out, alpha)
    idx = torch.arange(T) if idx is None else idx.long()
    src = torch.tensor(list(fin.chan_src))
    g = frames[:, idx][..., src].long()
    x = torch.stack([fin.lut32[c][g[..., c]] for c in range(C)], dim=1)          # (B, C, t, H0, W0)
    if tabs.resize:
        yi, yw, xi, xw = tabs.tables
        planes = x.reshape(-1, H0, W0).numpy()
        x = torch.from_numpy(_emulate_resize(planes, yi, yw, xi, xw)).reshape(B, C, t_out, tabs.Hr, tabs.Wr)
    rows = []
    for b in range(B):
        for v in range(len(views)):
            y0, x0 = tabs.crop_yx[2 * v], tabs.crop_yx[2 * v + 1]
            rows.append(x[b, :, :, y0:y0 + size, x0:x0 + size])
    return torch.stack(rows).contiguous()


@pytest.mark.parametrize("H0,W0,S,views,reverse,single", [
    (120, 160, 112, (0, 1, 2), False, False), (160, 120, 112, (2, 0, 1), True, False),
    (112, 149, 112, (0, 1, 2), False, False), (128, 171, 112, (1,), False, True), (120, 120, 112, (0, 2), True, False)])
def test_host_route_reproduces_oracle_rows(H0, W0, S, views, reverse, single):
    """Tables, crop offsets, channel map and frame index handed to the kernels reproduce the oracle's loader output --
    row order b * V + v included -- bit for bit when the kernel is emulated on the CPU."""
    g = torch.Generator().manual_seed(3)
    B, T, alpha = 2, 4, 4
    fr = torch.randint(0, 256, (B, T, H0, W0, 3), generator=g, dtype=torch.uint8)
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    cfg = helpers.case_cfg("slow_r50" if single else "dual_r50")
    cfg.DATA.MEAN, cfg.DATA.STD, cfg.DATA.REVERSE_INPUT_CHANNEL = mean, std, reverse
    fin = FR.FrameInput(cfg, torch.device("cpu"), torch.float16)
    want = SO.frames_to_crop_inputs(fr, mean, std, 1 if single else alpha, S, views, single, reverse)
    shapes = FR.view_shapes(fr.shape, S, views, None if single else alpha)
    assert [tuple(w.shape) for w in want] == shapes
    for w in want:
        assert torch.equal(_emulate_crop_route(fin, fr, S, views, w.shape[2], alpha), w)
    # the oracle's rows: clip b, view v at row b * V + v
    one = SO.frames_to_crop_inputs(fr[1:2], mean, std, 1 if single else alpha, S, views[-1:], single, reverse)
    assert torch.equal(want[-1][-1], one[-1][0])


def test_spatial_views_and_view_shapes_validate():
    assert FR.spatial_views(1) == (1,)
    assert FR.spatial_views([0, 1, 2]) == (0, 1, 2)
    assert FR.spatial_views(range(3)) == (0, 1, 2)
    for bad in (3, -1, (0, 3), (), [0] * 9, 1.0, True, "1", (None,), torch.tensor([2, 0])):
        with pytest.raises(ValueError):
            FR.spatial_views(bad)
    assert FR.view_shapes((2, 32, 256, 340, 3), 224, (0, 1, 2), 4) == [(6, 3, 8, 224, 224), (6, 3, 32, 224, 224)]
    assert FR.view_shapes((2, 8, 340, 256, 1), 224, 1) == [(2, 1, 8, 224, 224)]
    for size in (0, -4):
        with pytest.raises(ValueError):
            FR.view_shapes((1, 8, 64, 64, 3), size, 1)


def test_forward_frames_rejects_bad_crop_arguments_before_launch():
    """ValueError before anything reaches the device: CPU frames would otherwise be refused as not on the GPU."""
    cfg, model, _ = helpers.case_model_and_weights("dual_r50")
    model = model.eval()
    fr = torch.zeros(1, 32, 72, 96, 3, dtype=torch.uint8)
    for kw in (dict(spatial_idx=3), dict(spatial_idx=(0, 1, 5)), dict(spatial_idx=()), dict(crop_size=0),
               dict(spatial_idx=1, crop_size=-8)):
        with pytest.raises(ValueError):
            model.forward_frames(fr, **kw)
    with pytest.raises(ValueError):
        model.forward_frames(fr, bboxes=torch.zeros(1, 5), spatial_idx=1)
    with pytest.raises(Exception) as e:
        model.forward_frames(fr, spatial_idx=(0, 1, 2))               # valid arguments: refused only for the device
    assert not isinstance(e.value, ValueError)


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not mounted (ESF_REFERENCE_ROOT)")
def test_oracle_matches_reference_spatial_sampling():
    U = ref_shim.reference_dataset_utils()
    Tr = importlib.import_module("slowfast.datasets.transform")
    g = torch.Generator().manual_seed(21)
    for H0, W0, S in GEOMETRIES[:8]:
        x = torch.randn(4, H0, W0, 3, generator=g).permute(3, 0, 1, 2)
        for idx in (0, 1, 2):
            want = U.spatial_sampling(x, spatial_idx=idx, min_scale=S, max_scale=S, crop_size=S)
            assert torch.equal(SO.spatial_sampling(x, idx, S), want)
        r, _ = Tr.random_short_side_scale_jitter(x, S, S)
        assert torch.equal(SO.random_short_side_scale_jitter(x, S), r)
        for idx in (0, 1, 2):
            c, _ = Tr.uniform_crop(r, S, idx)
            assert torch.equal(SO.uniform_crop(r, S, idx), c)
    fr = torch.randint(0, 256, (5, 30, 40, 3), generator=g, dtype=torch.uint8)
    mean, std = [0.45] * 3, [0.225] * 3
    f = IO.tensor_normalize(fr, mean, std).permute(3, 0, 1, 2)
    assert torch.equal(U.spatial_sampling(f, spatial_idx=2, min_scale=32, max_scale=32, crop_size=32),
                       SO.frames_to_crop_inputs(fr[None], mean, std, 1, 32, (2,), True)[0][0])
