"""Test-time crops of clips of mixed decode sizes (forward_frames / ClipStream on a list of uint8 clips), host side:
clip-list shapes, argument validation before any launch, the staging arena's layout, and the error codes of the ragged
C entry points.  No GPU needed."""
import ctypes

import pytest
import torch

import helpers
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt


def test_view_shapes_of_a_clip_list():
    shapes = [(32, 256, 340, 3), (32, 340, 256, 3), (32, 720, 1280, 3)]
    assert FR.view_shapes(shapes, 224, (0, 1, 2)) == [(9, 3, 32, 224, 224)]
    assert FR.view_shapes(shapes, 224, (0, 1, 2), alpha=4) == [(9, 3, 8, 224, 224), (9, 3, 32, 224, 224)]
    # a list of clips of one size gives the shapes of the stacked batch (one plan for both)
    assert FR.view_shapes([(8, 120, 160, 3)] * 2, 112, 1, 4) == FR.view_shapes((2, 8, 120, 160, 3), 112, 1, 4)
    assert FR.view_shapes([torch.Size([8, 100, 100, 1])], 112, [1]) == [(1, 1, 8, 112, 112)]
    # the batch shape may still be given as a list of ints
    assert FR.view_shapes([2, 8, 120, 160, 3], 112, 1) == FR.view_shapes((2, 8, 120, 160, 3), 112, 1)


@pytest.mark.parametrize("shapes,size", [
    ([(8, 120, 160, 3), (4, 120, 160, 3)], 112),          # mixed T
    ([(8, 120, 160, 3), (8, 120, 160, 1)], 112),          # mixed C
    ([(1, 8, 120, 160, 3)], 112),                         # a stacked batch inside the list
    ([(8, 120, 160)], 112),                               # rank 3
    ([(8, 120, 160, 3), (8, 64, 64, 3)], 0),              # no crop of size 0 fits
    ([(8, 120, 160, 3), (8, 0, 64, 3)], 112),             # an empty clip
    ([(8, 120, 6000, 3)], 112),                           # rows of 18000 bytes
    ([], 112),
])
def test_view_shapes_rejects_bad_clip_lists(shapes, size):
    with pytest.raises(ValueError):
        FR.view_shapes(shapes, size, (0, 1, 2))


def test_arena_layout_aligns_every_clip():
    shapes = [(3, 5, 7, 3), (2, 4, 4, 1), (1, 1, 1, 1), (2, 8, 8, 3)]
    offsets, total = FR.arena_layout(shapes)
    sizes = [315, 32, 1, 384]
    assert offsets == [0, 320, 352, 368]
    assert total == 368 + 384
    for o, n, nxt in zip(offsets, sizes, offsets[1:] + [total]):
        assert o % 16 == 0 and o + n <= nxt
    assert FR.arena_layout(shapes, capacity=total) == (offsets, total)
    with pytest.raises(rt.EsfError):
        FR.arena_layout(shapes, capacity=total - 1)
    assert FR.arena_layout([]) == ([], 0)
    # B clips of the staging batch's own size always fit its B * T * H * W * C bytes when a clip is a multiple of 16
    assert FR.arena_layout([(8, 120, 160, 3)] * 4, capacity=4 * 8 * 120 * 160 * 3)[1] == 4 * 8 * 120 * 160 * 3


def test_forward_frames_rejects_bad_clip_lists_before_launch():
    """ValueError before anything reaches the device: CPU clips are otherwise refused as not on the GPU (EsfError)."""
    cfg, model, _ = helpers.case_model_and_weights("dual_r50")
    model = model.eval()
    a = torch.zeros(32, 72, 96, 3, dtype=torch.uint8)
    b = torch.zeros(32, 96, 72, 3, dtype=torch.uint8)
    bad_lists = [
        [a, torch.zeros(16, 72, 96, 3, dtype=torch.uint8)],             # mixed T
        [a, torch.zeros(32, 72, 96, 1, dtype=torch.uint8)],             # mixed C
        [a, torch.zeros(1, 32, 72, 96, 3, dtype=torch.uint8)],          # wrong rank
        [a, b.float()],                                                 # not uint8
        [a, torch.zeros(32, 96, 72, 6, dtype=torch.uint8)[..., :3]],   # not contiguous
        [a, torch.zeros(32, 72, 6000, 3, dtype=torch.uint8)],           # rows wider than 16384 bytes
        [a, "clip"],
    ]
    for clips in bad_lists:
        with pytest.raises(ValueError):
            model.forward_frames(clips, crop_size=64, spatial_idx=(0, 1, 2))
    for kw in (dict(spatial_idx=3), dict(spatial_idx=()), dict(crop_size=0), dict(crop_size=-8, spatial_idx=1),
               dict(bboxes=torch.zeros(1, 5)), dict(frame_index=[torch.zeros(8, dtype=torch.int32)] * 2)):
        with pytest.raises(ValueError):
            model.forward_frames([a, b], **{"crop_size": 64, **kw})
    with pytest.raises(Exception) as e:
        model.forward_frames((a, b), crop_size=64, spatial_idx=(0, 1, 2))     # valid: refused only for the device
    assert not isinstance(e.value, ValueError)
    with pytest.raises(Exception) as e:
        model.forward_frames([a, b])              # defaults of crop mode: DATA.TEST_CROP_SIZE, view 1
    assert not isinstance(e.value, ValueError)
    y = model.forward_frames([], crop_size=64, spatial_idx=(0, 1, 2))
    assert y.shape == (0, int(cfg.MODEL.NUM_CLASSES))


def _ragged_args(B=2, V=3, S=64, geom=None, crop=None, tables=True):
    """Arguments of esf_frames_to_clip_crop_ragged with fake device addresses: every call here must fail validation,
    i.e. before anything dereferences them or launches."""
    geom = geom or [(72, 96, 64, 85)] * B
    frames = (ctypes.c_void_p * B)(*[0x10000 * (b + 1) for b in range(B)])
    g = (ctypes.c_int32 * (4 * B))(*[n for gm in geom for n in gm])
    tabs = (ctypes.c_void_p * (4 * B))(*([0x900000 + 64 * i for i in range(4 * B)] if tables else [None] * (4 * B)))
    crop = crop or [(0, 0), (0, 10), (0, 21)] * B
    yx = (ctypes.c_int32 * (2 * V * B))(*[o for c in crop for o in c])
    return frames, B, 32, 3, None, 32, None, 0x800000, g, tabs, yx, V, S


def test_ragged_entry_points_reject_bad_arguments(esf_lib):
    L = esf_lib
    clip = 0x1000000
    n0 = rt.launch_count()
    ok = _ragged_args()
    bad = _ragged_args
    cases = [
        [None] + list(ok[1:]),                                             # no clip addresses
        list(ok[:1]) + [0] + list(ok[2:]),                                 # B = 0
        list(ok[:11]) + [9] + list(ok[12:]),                               # V > 8
        list(ok[:7]) + [None] + list(ok[8:]),                              # no lut
        list(ok[:4]) + [None, 8] + list(ok[6:]),                           # T != Tsrc without a frame index
        bad(crop=[(0, 0), (0, 10), (0, 21), (0, 0), (0, 10), (0, 22)]),    # clip 1's last crop leaves the frame
        bad(geom=[(72, 96, 64, 85), (72, 6000, 64, 5333)]),                # clip 1: rows of 18000 bytes
        bad(tables=False),                                                 # resized clips without tables
        bad(geom=[(72, 96, 64, 85), (0, 96, 64, 85)]),                     # clip 1: empty frame
    ]
    for args in cases:
        assert L.esf_frames_to_clip_crop_ragged(*args, clip, None) != 0
        assert L.esf_stem_pack_u8_crop_ragged(*args, rt.F16, 200, 3, clip, None) != 0
    assert L.esf_frames_to_clip_crop_ragged(*cases[5], clip, None) != 0
    msg = L.esf_last_error()
    assert b"clip 1" in msg and b"crop 2" in msg, msg
    # output checks: null / misaligned clip, bad dtype, pitch shorter than a row
    assert L.esf_frames_to_clip_crop_ragged(*ok, None, None) != 0
    assert L.esf_frames_to_clip_crop_ragged(*ok, clip + 4, None) != 0
    assert L.esf_stem_pack_u8_crop_ragged(*ok, rt.F32, 200, 3, clip, None) != 0
    assert L.esf_stem_pack_u8_crop_ragged(*ok, rt.F16, 192, 3, clip, None) != 0
    assert rt.launch_count() == n0      # every call was refused before the first launch
