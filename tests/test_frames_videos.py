"""Test-time temporal views of whole videos (forward_videos / ClipStream video mode), host side: the frame tables
against the CPU restatement of the reference's decoder (tests/temporal_oracle.py) and, where it is mounted, the
reference's own functions; the slow pathway's tables; row order, clip ids and view defaults; argument validation before
any launch; the error codes of the esf_*_crop_videos entry points.  No GPU needed."""
import ctypes
import importlib

import pytest
import torch

import helpers
import temporal_oracle as TO
from efficient_slowfast_b200 import config as esf_config
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.testing import TestMeter
from oracle import input_oracle as IO
from oracle import ref_shim

LENGTHS = [1, 20, 63, 64, 65, 300, 301]
RATES = [30, 25, 29.97, 60, 12]
NUM_CLIPS = [1, 2, 10]
# (NUM_FRAMES, SAMPLING_RATE, ALPHA) of the BASELINE models' test loaders: SlowFast 4x16 R50, SlowFast(-DA) 8x8 R50,
# the efficient 8x8 backbones as configured here (16 frames), Slow 8x8 R50 (single pathway)
TEMPORAL = [(32, 2, 8), (32, 2, 4), (16, 8, 4), (8, 8, None)]


def test_target_fps_default():
    assert esf_config.get_cfg().DATA.TARGET_FPS == 30


@pytest.mark.parametrize("T,rate,alpha", TEMPORAL)
def test_frame_tables_equal_oracle(T, rate, alpha):
    clamped = 0
    for N in LENGTHS:
        for fps in RATES:
            for nc in NUM_CLIPS:
                tabs = FR.video_frame_tables(N, fps, T, rate, 30, nc, alpha)
                fast = tabs[-1]
                assert fast.dtype == torch.int32 and fast.shape == (nc, T)
                for j in range(nc):
                    want = TO.sampled_index(N, rate, T, j, nc, fps, 30)
                    assert torch.equal(FR.temporal_index(N, fps, T, rate, 30, j, nc), want)
                    assert torch.equal(fast[j].long(), want)
                    assert int(fast[j].min()) >= 0 and int(fast[j].max()) <= N - 1
                    clamped += int(rate * T / 30 * fps > N)
    assert clamped > 0      # videos shorter than a clip are part of the grid


@pytest.mark.parametrize("T,rate,alpha", [t for t in TEMPORAL if t[2] is not None])
def test_slow_tables_equal_pack_pathway_output(T, rate, alpha):
    """The slow table is what pack_pathway_output makes of the sampled clip: frames that carry their own number."""
    for N in (20, 64, 301):
        video = torch.arange(N, dtype=torch.float32).view(N, 1, 1, 1).expand(N, 2, 2, 3).contiguous()
        for fps in (25, 29.97):
            slow, fast = FR.video_frame_tables(N, fps, T, rate, 30, 10, alpha)
            assert slow.shape == (10, T // alpha)
            for j, clip in enumerate(TO.view_clips(video, rate, T, 10, fps)):
                s, f = IO.pack_pathway_output(clip.permute(3, 0, 1, 2), alpha)
                assert torch.equal(f[0, :, 0, 0].long(), fast[j].long())
                assert torch.equal(s[0, :, 0, 0].long(), slow[j].long())


def test_frame_tables_are_cached_per_video_length_and_rate():
    fin = FR.FrameInput(esf_config.get_cfg(), torch.device("cpu"), torch.float16)
    a = fin.video_tables(300, 30.0, 32, 2, 30, 10, 4)
    assert fin.video_tables(300, 30.0, 32, 2, 30, 10, 4) is a
    assert fin.video_tables(301, 30.0, 32, 2, 30, 10, 4) is not a


@pytest.mark.skipif(not ref_shim.available(), reason="reference tree not mounted (ESF_REFERENCE_ROOT)")
def test_oracle_matches_reference_decoder():
    ref_shim.reference_dataset_utils()
    D = importlib.import_module("slowfast.datasets.decoder")
    for N in LENGTHS:
        for fps in RATES:
            for T, rate, _ in TEMPORAL:
                clip_sz = rate * T / 30 * fps
                for nc in NUM_CLIPS:
                    for j in range(nc):
                        want = D.get_start_end_idx(N, clip_sz, j, nc)
                        assert TO.get_start_end_idx(N, clip_sz, j, nc) == tuple(want)[:2]
                        frames = torch.arange(N)
                        assert torch.equal(TO.temporal_sampling(frames, *want[:2], T),
                                           D.temporal_sampling(frames, *want[:2], T))


def test_view_defaults_and_row_order():
    assert FR.ensemble_spatial_views(3) == (0, 1, 2)
    assert FR.ensemble_spatial_views(2) == (0, 1)
    assert FR.ensemble_spatial_views(1) == (1,)
    with pytest.raises(ValueError):
        FR.ensemble_spatial_views(0)
    # a VideoList's clip b is video b // num_clips at temporal view b % num_clips, tables in that order
    videos = [torch.zeros(n, h, w, 3, dtype=torch.uint8) for n, h, w in ((40, 72, 96), (300, 96, 72), (7, 64, 64))]
    fps = [30.0, 25.0, 12.0]
    views, nc = (0, 1, 2), 10
    crops = [FR.CropTables(v.shape[1], v.shape[2], 64, views, "cpu") for v in videos]
    tables = [FR.video_frame_tables(v.shape[0], f, 32, 2, 30, nc, 4) for v, f in zip(videos, fps)]
    vl = FR.VideoList(videos, crops, tables, nc)
    assert (vl.B, vl.V, vl.T) == (30, 3, [8, 32])
    for b in range(vl.B):
        v = b // nc
        assert vl.frames[b] == videos[v].data_ptr()
        assert list(vl.geom[5 * b:5 * b + 5]) == [videos[v].shape[0], crops[v].H0, crops[v].W0, crops[v].Hr,
                                                   crops[v].Wr]
        assert list(vl.crop_yx[6 * b:6 * b + 6]) == list(crops[v].crop_yx)
    slow = vl.index[:vl.B * 8].view(vl.B, 8)
    fast = vl.index[vl.B * 8:].view(vl.B, 32)
    for b in range(vl.B):
        assert torch.equal(slow[b], tables[b // nc][0][b % nc]) and torch.equal(fast[b], tables[b // nc][1][b % nc])
    # row (v * nc + j) * V + s is the test loader's clip v * nc * V + (j * V + s): temporal j = idx // V, crop idx % V
    V = len(views)
    for v in range(3):
        for idx in range(nc * V):
            j, s = idx // V, idx % V
            assert (v * nc + j) * V + s == v * nc * V + idx
    # TestMeter(num_clips = nc * V) gathers the rows of a video by clip id // (nc * V)
    meter = TestMeter(3, nc * V, 4, 1)
    rows = torch.arange(3 * nc * V * 4, dtype=torch.float32).view(-1, 4)
    meter.update_stats(rows, torch.tensor([1, 2, 3]).repeat_interleave(nc * V), torch.arange(3 * nc * V))
    assert torch.equal(meter.video_preds, rows.view(3, nc * V, 4).sum(1))
    assert meter.clip_count.tolist() == [nc * V] * 3


def _videos(*shapes, dtype=torch.uint8):
    return [torch.zeros(s, dtype=dtype) for s in shapes]


def test_forward_videos_rejects_bad_arguments_before_launch():
    """ValueError before anything reaches the device: CPU videos are otherwise refused as not on the GPU (EsfError)."""
    cfg, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.eval()
    a, b = _videos((40, 72, 96, 3), (25, 96, 72, 3))
    bad_lists = [
        [a, torch.zeros(25, 96, 72, 1, dtype=torch.uint8)],               # mixed C
        [a, torch.zeros(0, 96, 72, 3, dtype=torch.uint8)],                # N_v = 0
        [a, torch.zeros(1, 25, 96, 72, 3, dtype=torch.uint8)],            # wrong rank
        [a, b.float()],                                                   # not uint8
        [a, torch.zeros(25, 96, 72, 6, dtype=torch.uint8)[..., :3]],     # not contiguous
        [a, torch.zeros(25, 72, 6000, 3, dtype=torch.uint8)],             # rows wider than 16384 bytes
        [a, "video"],
    ]
    for videos in bad_lists:
        with pytest.raises(ValueError):
            model.forward_videos(videos, crop_size=64)
    for kw in (dict(fps=0), dict(fps=-25.0), dict(fps=[30, 0]), dict(fps=[30]), dict(fps=float("nan")),
               dict(num_clips=0), dict(num_clips=2.5), dict(spatial_idx=3), dict(spatial_idx=()),
               dict(crop_size=0), dict(crop_size=-8), dict(bboxes=torch.zeros(1, 5))):
        with pytest.raises(ValueError):
            model.forward_videos([a, b], **{"crop_size": 64, **kw})
    with pytest.raises(ValueError):
        model.forward_videos(a)                  # a tensor, not a list of videos
    with pytest.raises(Exception) as e:
        model.forward_videos((a, b), fps=[30, 25.0], crop_size=64, num_clips=2, spatial_idx=[0, 2])
    assert not isinstance(e.value, ValueError)   # valid: refused only for the device
    assert isinstance(e.value, rt.EsfError)
    with pytest.raises(Exception) as e:
        model.forward_videos([torch.zeros(40, 256, 340, 3, dtype=torch.uint8)])   # defaults: 10 x 3 views at 256
    assert not isinstance(e.value, ValueError)
    y = model.forward_videos([], crop_size=64)
    assert y.shape == (0, int(cfg.MODEL.NUM_CLASSES))


def _video_args(B=2, V=3, S=64, geom=None, crop=None, tables=True, t_index=0x700000):
    """Arguments of esf_frames_to_clip_crop_videos with fake device addresses: every call here must fail validation,
    i.e. before anything dereferences them or launches."""
    geom = geom or [(40, 72, 96, 64, 85)] * B
    frames = (ctypes.c_void_p * B)(*[0x10000 * (b // 2 + 1) for b in range(B)])
    g = (ctypes.c_int32 * (5 * B))(*[n for gm in geom for n in gm])
    tabs = (ctypes.c_void_p * (4 * B))(*([0x900000 + 64 * i for i in range(4 * B)] if tables else [None] * (4 * B)))
    crop = crop or [(0, 0), (0, 10), (0, 21)] * B
    yx = (ctypes.c_int32 * (2 * V * B))(*[o for c in crop for o in c])
    return frames, B, 3, t_index, 32, None, 0x800000, g, tabs, yx, V, S


def test_video_entry_points_reject_bad_arguments(esf_lib):
    L = esf_lib
    clip = 0x1000000
    n0 = rt.launch_count()
    ok = _video_args()
    bad = _video_args
    cases = [
        [None] + list(ok[1:]),                                                  # no video addresses
        list(ok[:1]) + [0] + list(ok[2:]),                                      # B = 0
        list(ok[:10]) + [9] + list(ok[11:]),                                    # V > 8
        list(ok[:6]) + [None] + list(ok[7:]),                                   # no lut
        bad(t_index=None),                                                      # no frame table
        bad(geom=[(40, 72, 96, 64, 85), (0, 72, 96, 64, 85)]),                  # clip 1: a video of no frames
        bad(crop=[(0, 0), (0, 10), (0, 21), (0, 0), (0, 10), (0, 22)]),         # clip 1's last crop leaves the frame
        bad(geom=[(40, 72, 96, 64, 85), (40, 72, 6000, 64, 5333)]),             # clip 1: rows of 18000 bytes
        bad(tables=False),                                                      # resized clips without tables
        bad(geom=[(40, 72, 96, 64, 85), (40, 0, 96, 64, 85)]),                  # clip 1: empty frame
    ]
    for args in cases:
        assert L.esf_frames_to_clip_crop_videos(*args, clip, None) != 0
        assert L.esf_stem_pack_u8_crop_videos(*args, rt.F16, 200, 3, clip, None) != 0
    assert L.esf_frames_to_clip_crop_videos(*cases[5], clip, None) != 0
    msg = L.esf_last_error()
    assert b"clip 1" in msg and b"0 frames" in msg, msg
    assert L.esf_stem_pack_u8_crop_videos(*cases[4], rt.F16, 200, 3, clip, None) != 0
    assert b"frame table" in L.esf_last_error()
    # output checks: null / misaligned clip, bad dtype, pitch shorter than a row
    assert L.esf_frames_to_clip_crop_videos(*ok, None, None) != 0
    assert L.esf_frames_to_clip_crop_videos(*ok, clip + 4, None) != 0
    assert L.esf_stem_pack_u8_crop_videos(*ok, rt.F32, 200, 3, clip, None) != 0
    assert L.esf_stem_pack_u8_crop_videos(*ok, rt.F16, 192, 3, clip, None) != 0
    assert rt.launch_count() == n0      # every call was refused before the first launch
