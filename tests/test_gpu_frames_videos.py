"""Test-time temporal views of whole videos (csrc/esf_crop.cu esf_*_crop_videos behind forward_videos and ClipStream
video mode) against the CPU restatement of the reference's test loader: temporal sampling of every view out of the
decoded video (tests/temporal_oracle.py), then the spatial chain of every clip (tests/spatial_oracle.py), rows
concatenated in the loader's clip order.  Every resized width here is >= 104, where the kernel reproduces torch's CPU
interpolate bit for bit (DESIGN 3.7), so every comparison is exact."""
import pytest
import torch

import helpers
import spatial_oracle as SO
import temporal_oracle as TO
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.testing import TestMeter

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
GUARD = 64   # sentinel elements after every output: the kernels must not write past their rows
# (frames, H, W, fps) at S = 112: landscape, portrait, crop only (short side already 112), identity, 16:9; lengths
# below one clip (clamped indices), around it and well above it
VIDEOS = [(45, 120, 160, 30.0), (9, 160, 120, 25.0), (130, 112, 150, 29.97), (64, 112, 112, 60.0),
          (33, 128, 171, 12.0)]


def _random_videos(spec, C, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, (N, H, W, C), generator=g, dtype=torch.uint8) for N, H, W, _ in spec]


def _oracle_clips(videos, rates, T, rate, nc):
    """The uint8 clips of every temporal view, in the loader's order (video, temporal view)."""
    return [c for v, f in zip(videos, rates) for c in TO.view_clips(v, rate, T, nc, f)]


def _oracle(clips, mean, std, alpha, S, views, single=False, reverse=False):
    per = [SO.frames_to_crop_inputs(c[None], mean, std, alpha, S, views, single, reverse) for c in clips]
    return [torch.cat([p[i] for p in per]) for i in range(len(per[0]))]


def _frame_input(C, reverse):
    cfg = helpers.case_cfg("dual_r50")
    cfg.DATA.MEAN, cfg.DATA.STD, cfg.DATA.REVERSE_INPUT_CHANNEL = MEAN[:C], STD[:C], reverse
    return FR.FrameInput(cfg, torch.device("cuda"), torch.float16, channels=C)


def _check_videos(L, fin, videos, rates, want, T, rate, alpha, nc, C, S, views):
    """Both video entry points == `want` (FP32 clips per pathway, and esf_stem_pack of them), bit for bit, nothing
    written past the outputs."""
    dev = [v.cuda() for v in videos]
    tables = [fin.video_tables(v.shape[0], f, T, rate, 30, nc, alpha) for v, f in zip(videos, rates)]
    batch = FR.VideoList(dev, [fin.crop(v.shape[1], v.shape[2], S, views) for v in videos], tables, nc)
    index = batch.index.cuda()
    s = rt.current_stream_ptr()
    pitch, lpad, _ = rt.stem_geometry(S, C, 7, 2, 3)
    off = 0
    for w, To in zip(want, batch.T):
        assert w.shape[0] == batch.B * batch.V and w.shape[2] == To
        args = (batch.frames, batch.B, C, index[off:].data_ptr(), To, fin.chan_src, fin.lut32.data_ptr(), batch.geom,
                batch.tables, batch.crop_yx, batch.V, S)
        off += batch.B * To
        out = torch.full((w.numel() + GUARD,), 7.0, device="cuda")
        rt.check(L.esf_frames_to_clip_crop_videos(*args, out.data_ptr(), s))
        wd = w.cuda()
        for dt in (torch.float16, torch.bfloat16):
            n = w.shape[0] * To * S * pitch
            a = torch.full((n,), 5, dtype=dt, device="cuda")
            b = torch.full((n + GUARD,), 9, dtype=dt, device="cuda")
            rt.check(L.esf_stem_pack(wd.data_ptr(), w.shape[0], C, To, S, S, pitch, lpad, rt.dtype_code(dt),
                                     a.data_ptr(), s))
            rt.check(L.esf_stem_pack_u8_crop_videos(*args, rt.dtype_code(dt), pitch, lpad, b.data_ptr(), s))
            torch.cuda.synchronize()
            assert torch.equal(a.view(torch.int16), b[:n].view(torch.int16))
            assert torch.equal(b[n:].float().cpu(), torch.full((GUARD,), 9.0))
        torch.cuda.synchronize()
        assert torch.equal(out[:w.numel()].cpu().view(w.shape), w)
        assert torch.equal(out[w.numel():].cpu(), torch.full((GUARD,), 7.0))


@pytest.mark.parametrize("C,reverse", [(3, False), (1, False), (3, True)])
def test_video_kernels_equal_oracle(esf_lib, C, reverse):
    """Videos of mixed length and size (landscape, portrait, crop only, identity), both pathways, grey and
    reversed-channel input, FP16 and BF16 packed rows; 5 videos x 2 temporal views."""
    T, rate, alpha, nc, S, views = 8, 4, 4, 2, 112, (0, 1, 2)
    videos = _random_videos(VIDEOS, C, 70 + C + reverse)
    rates = [f for *_, f in VIDEOS]
    want = _oracle(_oracle_clips(videos, rates, T, rate, nc), MEAN[:C], STD[:C], alpha, S, views, False, reverse)
    _check_videos(esf_lib, _frame_input(C, reverse), videos, rates, want, T, rate, alpha, nc, C, S, views)


def test_video_kernels_across_launch_chunks(esf_lib):
    """5 videos x 10 temporal views = 50 clips, more than one launch takes (32)."""
    T, rate, alpha, nc, S, views = 4, 8, 4, 10, 112, (0, 2)
    videos = _random_videos(VIDEOS, 3, 71)
    rates = [f for *_, f in VIDEOS]
    want = _oracle(_oracle_clips(videos, rates, T, rate, nc), MEAN, STD, alpha, S, views)
    _check_videos(esf_lib, _frame_input(3, False), videos, rates, want, T, rate, alpha, nc, 3, S, views)


@pytest.mark.parametrize("name,precision", [
    ("slowfast_r50", "fp16"), ("shufflenetv2_w05", "fp16"), ("slow_r50", "fp16"), ("slowfast_r50", "fp32")])
def test_forward_videos_equals_forward_frames_on_oracle_clips(esf_lib, name, precision):
    """forward_videos == forward_frames(list of the oracle's temporal clips), bit for bit, from the same plan."""
    cfg, model, _ = helpers.case_model_and_weights(name, precision)
    model = model.cuda().eval()
    S, views, nc = 112, (0, 1, 2), 2
    T, rate = int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.SAMPLING_RATE)
    spec = VIDEOS[:3]
    videos = _random_videos(spec, 3, 72)
    rates = [f for *_, f in spec]
    clips = [c.cuda() for c in _oracle_clips(videos, rates, T, rate, nc)]
    dev = [v.cuda() for v in videos]
    with torch.no_grad():
        y_ref = model.forward_frames(clips, crop_size=S, spatial_idx=views).cpu()
        plans = list(model._plans.values())
        y = model.forward_videos(dev, fps=rates, num_clips=nc, crop_size=S, spatial_idx=views).cpu()
        assert list(model._plans.values()) == plans      # no new plan: the forward_frames plan of 6 clips
        y2 = model.forward_videos(tuple(dev), fps=rates, num_clips=nc, crop_size=S, spatial_idx=list(views)).cpu()
    assert y.shape[0] == len(videos) * nc * len(views) and torch.isfinite(y).all()
    assert torch.equal(y, y_ref)
    assert torch.equal(y, y2)


def test_forward_videos_defaults(esf_lib):
    """TARGET_FPS, NUM_ENSEMBLE_VIEWS and NUM_SPATIAL_CROPS of the config: 2 videos x 10 x 3 rows."""
    cfg, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    S = 112
    T, rate = int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.SAMPLING_RATE)
    videos = _random_videos([(300, 112, 150, 30.0), (20, 150, 112, 30.0)], 3, 73)
    clips = [c.cuda() for c in _oracle_clips(videos, [30.0, 30.0], T, rate, 10)]
    with torch.no_grad():
        y = model.forward_videos([v.cuda() for v in videos], crop_size=S).cpu()
        y_ref = model.forward_frames(clips, crop_size=S, spatial_idx=(0, 1, 2)).cpu()
    assert y.shape[0] == 60
    assert torch.equal(y, y_ref)


def test_clipstream_video_mode_equals_forward_videos_and_testmeter(esf_lib):
    import efficient_slowfast_b200 as esf

    _, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    S, views, nc = 112, (0, 1, 2), 3
    cfg = model._cfg
    T, rate = int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.SAMPLING_RATE)
    st = esf.ClipStream(model, [(2, 64, 160, 160, 3)], frames=True, num_clips=nc, crop_size=S, spatial_idx=views)
    too_many_bytes = [v.pin_memory() for v in _random_videos([(64, 160, 200, 0), (64, 160, 160, 0)], 3, 74)]
    too_many_videos = [v.pin_memory() for v in _random_videos([(8, 112, 112, 0)] * 3, 3, 75)]
    for bad in (too_many_bytes, too_many_videos):
        with pytest.raises(rt.EsfError):
            st.submit(bad)
    with pytest.raises(ValueError):
        st.submit(too_many_videos[:2], fps=0)
    spec = [VIDEOS[:2], VIDEOS[2:4], VIDEOS[4:5]]      # the last batch is short
    batches = [[v.pin_memory() for v in _random_videos(sp, 3, 80 + i)] for i, sp in enumerate(spec)]
    rates = [[f for *_, f in sp] for sp in spec]
    got = []
    with torch.no_grad():
        for b, r in zip(batches, rates):
            out = st.submit(b, fps=r)
            if out is not None:
                got.append(out)
        got += st.flush()
        want = [model.forward_videos([v.cuda() for v in b], fps=r, num_clips=nc, crop_size=S,
                                     spatial_idx=views).cpu() for b, r in zip(batches, rates)]
        # the per-view route: host temporal sampling into uint8 clips, then a list of clips
        per_view = [model.forward_frames([c.cuda() for c in _oracle_clips(b, r, T, rate, nc)], crop_size=S,
                                         spatial_idx=views).cpu() for b, r in zip(batches, rates)]
    assert [i for i, _ in got] == [0, 1, 2]
    for (_, y), w, p, b in zip(got, want, per_view, batches):
        assert y.shape[0] == len(b) * nc * len(views)
        assert torch.equal(y, w)
        assert torch.equal(y, p)
    # TestMeter on the video-mode rows and on the per-view rows: the same video-level predictions (sum and max)
    K = nc * len(views)
    n_videos = sum(len(b) for b in batches)
    labels = torch.arange(n_videos) % 7 + 1
    for method in ("sum", "max"):
        meters = [TestMeter(n_videos, K, got[0][1].shape[1], 1, ensemble_method=method) for _ in range(2)]
        v0 = 0
        for (_, y), p, b in zip(got, per_view, batches):
            ids = v0 * K + torch.arange(y.shape[0])
            lab = labels[v0:v0 + len(b)].repeat_interleave(K)
            meters[0].update_stats(y, lab, ids)
            meters[1].update_stats(p, lab, ids)
            v0 += len(b)
        assert torch.equal(meters[0].video_preds, meters[1].video_preds)
        assert meters[0].clip_count.tolist() == [K] * n_videos
