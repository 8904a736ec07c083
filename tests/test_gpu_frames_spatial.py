"""Test-time spatial sampling on the device (csrc/esf_crop.cu behind forward_frames(crop_size=, spatial_idx=)) against
the CPU restatement of the reference's test loader (tests/spatial_oracle.py).  Every resized width here is >= 104, where
the kernel reproduces torch's CPU interpolate bit for bit (DESIGN 3.7), so every comparison is exact."""
import ctypes

import pytest
import torch

import helpers
import spatial_oracle as SO
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
GUARD = 64   # sentinel elements after every output: the kernels must not write past their rows


@pytest.mark.parametrize("H0,W0,S,C,reverse", [
    (256, 340, 224, 3, False), (340, 256, 224, 3, False), (240, 320, 224, 3, True), (720, 1280, 256, 3, False),
    (224, 298, 224, 3, False), (224, 224, 224, 3, False), (256, 340, 224, 1, False), (128, 171, 112, 3, True)])
def test_crop_kernels_equal_oracle(esf_lib, H0, W0, S, C, reverse):
    """FP32 clip and packed 16-bit rows of both pathways == the oracle's loader output (and esf_stem_pack of it), bit
    for bit, three views; nothing written past the outputs."""
    g = torch.Generator().manual_seed(H0 + W0 + C)
    B, T, alpha, views = 2, 8, 4, (0, 1, 2)
    fr = torch.randint(0, 256, (B, T, H0, W0, C), generator=g, dtype=torch.uint8)
    mean, std = MEAN[:C], STD[:C]
    want = SO.frames_to_crop_inputs(fr, mean, std, alpha, S, views, False, reverse)
    cfg = helpers.case_cfg("dual_r50")
    cfg.DATA.MEAN, cfg.DATA.STD, cfg.DATA.REVERSE_INPUT_CHANNEL = mean, std, reverse
    fin = FR.FrameInput(cfg, torch.device("cuda"), torch.float16, channels=C)
    tabs = fin.crop(H0, W0, S, views)
    geo = tabs.pointers() + (tabs.crop_yx, len(views), S)
    frd = fr.cuda()
    s = rt.current_stream_ptr()
    pitch, lpad, _ = rt.stem_geometry(S, C, 7, 2, 3)
    for w in want:
        To = w.shape[2]
        idx = fin.index(T, To, alpha)
        iptr = idx.data_ptr() if idx is not None else None
        out = torch.full((w.numel() + GUARD,), 7.0, device="cuda")
        rt.check(esf_lib.esf_frames_to_clip_crop(frd.data_ptr(), B, T, H0, W0, C, iptr, To, fin.chan_src,
                                                 fin.lut32.data_ptr(), *geo, out.data_ptr(), s))
        for dt in (torch.float16, torch.bfloat16):
            n = B * len(views) * To * S * pitch
            a = torch.full((n,), 5, dtype=dt, device="cuda")
            b = torch.full((n + GUARD,), 9, dtype=dt, device="cuda")
            wd = w.cuda()
            rt.check(esf_lib.esf_stem_pack(wd.data_ptr(), w.shape[0], C, To, S, S, pitch, lpad, rt.dtype_code(dt),
                                           a.data_ptr(), s))
            rt.check(esf_lib.esf_stem_pack_u8_crop(frd.data_ptr(), B, T, H0, W0, C, iptr, To, fin.chan_src,
                                                   fin.lut32.data_ptr(), *geo, rt.dtype_code(dt), pitch, lpad,
                                                   b.data_ptr(), s))
            torch.cuda.synchronize()
            assert torch.equal(a.view(torch.int16), b[:n].view(torch.int16))
            assert torch.equal(b[n:].float().cpu(), torch.full((GUARD,), 9.0))
        torch.cuda.synchronize()
        assert torch.equal(out[:w.numel()].cpu().view(w.shape), w)
        assert torch.equal(out[w.numel():].cpu(), torch.full((GUARD,), 7.0))
        if (H0, W0) == (S, S):           # identity geometry: the crop route equals today's route bit for bit
            old = torch.empty((B,) + tuple(w.shape[1:]), device="cuda")
            rt.check(esf_lib.esf_frames_to_clip(frd.data_ptr(), B, T, H0, W0, C, iptr, To, fin.chan_src,
                                                fin.lut32.data_ptr(), old.data_ptr(), s))
            torch.cuda.synchronize()
            assert torch.equal(old.cpu().repeat_interleave(len(views), 0), w)


def test_crop_kernels_reject_bad_arguments(esf_lib):
    fr = torch.zeros(1, 4, 64, 80, 3, dtype=torch.uint8, device="cuda")
    lut = torch.zeros(3, 256, device="cuda")
    out = torch.zeros(1 << 20, device="cuda")
    s = rt.current_stream_ptr()
    yx = (ctypes.c_int32 * 2)(0, 17)          # 64-wide crop at x0 = 17 leaves an 80-wide frame
    assert esf_lib.esf_frames_to_clip_crop(fr.data_ptr(), 1, 4, 64, 80, 3, None, 4, None, lut.data_ptr(), None, None,
                                           64, None, None, 80, yx, 1, 64, out.data_ptr(), s) != 0
    yx = (ctypes.c_int32 * 2)(0, 8)
    assert esf_lib.esf_frames_to_clip_crop(fr.data_ptr(), 1, 4, 64, 80, 3, None, 4, None, lut.data_ptr(), None, None,
                                           56, None, None, 70, yx, 1, 56, out.data_ptr(), s) != 0   # resize, no tables
    assert esf_lib.esf_frames_to_clip_crop(fr.data_ptr(), 1, 4, 64, 80, 3, None, 4, None, lut.data_ptr(), None, None,
                                           64, None, None, 80, yx, 9, 64, out.data_ptr(), s) != 0   # V > 8


@pytest.mark.parametrize("name,frames,H0,W0,S", [
    ("slowfast_r50", 32, 120, 160, 112), ("dual_r50", 32, 160, 120, 112), ("shufflenetv2_w05", 16, 128, 171, 112),
    ("slow_r50", 8, 120, 160, 112), ("slowfast_r50", 32, 256, 340, 256)])   # last: crop only, fully-convolutional head
def test_forward_frames_crops_equal_forward_on_oracle_clips(esf_lib, name, frames, H0, W0, S):
    cfg, model, _ = helpers.case_model_and_weights(name)
    model = model.cuda().eval()
    g = torch.Generator().manual_seed(40)
    fr = torch.randint(0, 256, (1, frames, H0, W0, 3), generator=g, dtype=torch.uint8)
    single = model.num_pathways == 1
    xs = SO.frames_to_crop_inputs(fr, cfg.DATA.MEAN, cfg.DATA.STD, 1 if single else cfg.SLOWFAST.ALPHA, S, (0, 1, 2),
                                  single, False)
    with torch.no_grad():
        y_ref = model([t.cuda() for t in xs]).cpu()
        y = model.forward_frames(fr.cuda(), crop_size=S, spatial_idx=(0, 1, 2)).cpu()
        y2 = model.forward_frames(fr.cuda(), crop_size=S, spatial_idx=[0, 1, 2]).cpu()     # graph replay
        y1 = model.forward_frames(fr.cuda(), crop_size=S, spatial_idx=2).cpu()
    assert y.shape[0] == 3 and torch.isfinite(y).all()
    assert torch.equal(y.argmax(1), y_ref.argmax(1))
    assert torch.equal(y, y_ref)
    assert torch.equal(y, y2)
    assert torch.equal(y1.argmax(1), y[2:].argmax(1))       # view 2 alone (a plan for one row)
    with pytest.raises(ValueError):
        model.forward_frames(fr.cuda(), spatial_idx=(0, 3))


def test_clipstream_crop_mode_equals_forward_frames(esf_lib):
    import efficient_slowfast_b200 as esf

    cfg, model, _ = helpers.case_model_and_weights("dual_r50")
    model = model.cuda().eval()
    g = torch.Generator().manual_seed(41)
    batches = [torch.randint(0, 256, (2, 32, 120, 160, 3), generator=g, dtype=torch.uint8).pin_memory()
               for _ in range(3)]
    st = esf.ClipStream(model, [tuple(batches[0].shape)], frames=True, crop_size=112, spatial_idx=(0, 1, 2))
    got = []
    with torch.no_grad():
        for b in batches:
            r = st.submit([b])
            if r is not None:
                got.append(r)
        got += st.flush()
        want = [model.forward_frames(b.cuda(), crop_size=112, spatial_idx=(0, 1, 2)).cpu() for b in batches]
    assert [i for i, _ in got] == [0, 1, 2]
    for (_, y), w in zip(got, want):
        assert y.shape[0] == 6
        assert torch.equal(y, w)
    assert st.h2d_bytes == 2 * 32 * 120 * 160 * 3
