"""Test-time crops of clips of mixed decode sizes (csrc/esf_crop.cu esf_*_crop_ragged behind forward_frames(list) and
ClipStream) against the CPU restatement of the reference's test loader, run on every clip alone (tests/spatial_oracle.py)
with the rows concatenated, as the collate function does.  Every resized width here is >= 104, where the kernel
reproduces torch's CPU interpolate bit for bit (DESIGN 3.7), so every comparison is exact."""
import pytest
import torch

import helpers
import spatial_oracle as SO
from efficient_slowfast_b200 import frames as FR
from efficient_slowfast_b200 import runtime as rt

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
GUARD = 64   # sentinel elements after every output: the kernels must not write past their rows
# landscape, portrait, 720p, crop only (short side already 224), identity, 4:3 -- one clip each
GEOMETRIES = [(256, 340), (340, 256), (720, 1280), (224, 298), (224, 224), (240, 320)]
# S = 112: landscape, portrait, crop only, identity, 16:9
SMALL = [(120, 160), (160, 120), (112, 150), (112, 112), (128, 171)]


def _oracle(clips, mean, std, alpha, S, views, single=False, reverse=False):
    per = [SO.frames_to_crop_inputs(c[None], mean, std, alpha, S, views, single, reverse) for c in clips]
    return [torch.cat([p[i] for p in per]) for i in range(len(per[0]))]


def _frame_input(C, reverse):
    cfg = helpers.case_cfg("dual_r50")
    cfg.DATA.MEAN, cfg.DATA.STD, cfg.DATA.REVERSE_INPUT_CHANNEL = MEAN[:C], STD[:C], reverse
    return FR.FrameInput(cfg, torch.device("cuda"), torch.float16, channels=C)


def _random_clips(sizes, T, C, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, 256, (T, H, W, C), generator=g, dtype=torch.uint8) for H, W in sizes]


def _check_ragged(L, fin, clips, want, T, alpha, C, S, views):
    """Both ragged entry points on `clips` == `want` (FP32 clips per pathway, and esf_stem_pack of them), bit for bit,
    nothing written past the outputs."""
    dev = [c.cuda() for c in clips]
    batch = FR.ClipList(dev, [fin.crop(c.shape[1], c.shape[2], S, views) for c in clips])
    s = rt.current_stream_ptr()
    pitch, lpad, _ = rt.stem_geometry(S, C, 7, 2, 3)
    for w in want:
        To = w.shape[2]
        idx = fin.index(T, To, alpha)
        args = (batch.frames, batch.B, T, C, idx.data_ptr() if idx is not None else None, To, fin.chan_src,
                fin.lut32.data_ptr(), batch.geom, batch.tables, batch.crop_yx, batch.V, S)
        out = torch.full((w.numel() + GUARD,), 7.0, device="cuda")
        rt.check(L.esf_frames_to_clip_crop_ragged(*args, out.data_ptr(), s))
        wd = w.cuda()
        for dt in (torch.float16, torch.bfloat16):
            n = w.shape[0] * To * S * pitch
            a = torch.full((n,), 5, dtype=dt, device="cuda")
            b = torch.full((n + GUARD,), 9, dtype=dt, device="cuda")
            rt.check(L.esf_stem_pack(wd.data_ptr(), w.shape[0], C, To, S, S, pitch, lpad, rt.dtype_code(dt),
                                     a.data_ptr(), s))
            rt.check(L.esf_stem_pack_u8_crop_ragged(*args, rt.dtype_code(dt), pitch, lpad, b.data_ptr(), s))
            torch.cuda.synchronize()
            assert torch.equal(a.view(torch.int16), b[:n].view(torch.int16))
            assert torch.equal(b[n:].float().cpu(), torch.full((GUARD,), 9.0))
        torch.cuda.synchronize()
        assert torch.equal(out[:w.numel()].cpu().view(w.shape), w)
        assert torch.equal(out[w.numel():].cpu(), torch.full((GUARD,), 7.0))


@pytest.mark.parametrize("C,reverse", [(3, False), (1, False), (3, True)])
def test_ragged_kernels_equal_per_clip_oracle(esf_lib, C, reverse):
    """One batch of landscape, portrait, 720p, crop-only and identity clips; both pathways (the slow one through the
    frame index), grey and reversed-channel variants, FP16 and BF16 packed rows."""
    T, alpha, S, views = 8, 4, 224, (0, 1, 2)
    clips = _random_clips(GEOMETRIES, T, C, 50 + C + reverse)
    want = _oracle(clips, MEAN[:C], STD[:C], alpha, S, views, False, reverse)
    _check_ragged(esf_lib, _frame_input(C, reverse), clips, want, T, alpha, C, S, views)


def test_ragged_kernels_across_launch_chunks(esf_lib):
    """More clips than one launch takes (32): the chunk boundaries keep the row order and write nothing twice."""
    T, alpha, S, views = 4, 4, 112, (0, 2)
    clips = _random_clips([SMALL[i % len(SMALL)] for i in range(70)], T, 3, 51)
    want = _oracle(clips, MEAN, STD, alpha, S, views)
    _check_ragged(esf_lib, _frame_input(3, False), clips, want, T, alpha, 3, S, views)


def test_one_size_list_equals_stacked_route(esf_lib):
    """A list of clips of one size and the stacked tensor of them: the same kernel output and the same predictions,
    bit for bit, from the same plan."""
    T, S, views = 4, 112, (0, 1, 2)
    fr = torch.stack(_random_clips([(128, 171)] * 34, T, 3, 52)).cuda()
    fin = _frame_input(3, False)
    tabs = fin.crop(128, 171, S, views)
    batch = FR.ClipList(list(fr), [tabs] * fr.shape[0])
    s = rt.current_stream_ptr()
    n = fr.shape[0] * len(views) * 3 * T * S * S
    a, b = torch.zeros(n, device="cuda"), torch.ones(n, device="cuda")
    rt.check(esf_lib.esf_frames_to_clip_crop(fr.data_ptr(), fr.shape[0], T, 128, 171, 3, None, T, fin.chan_src,
                                             fin.lut32.data_ptr(), *tabs.pointers(), tabs.crop_yx, len(views), S,
                                             a.data_ptr(), s))
    rt.check(esf_lib.esf_frames_to_clip_crop_ragged(batch.frames, batch.B, T, 3, None, T, fin.chan_src,
                                                    fin.lut32.data_ptr(), batch.geom, batch.tables, batch.crop_yx,
                                                    len(views), S, b.data_ptr(), s))
    torch.cuda.synchronize()
    assert torch.equal(a, b)

    _, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    fr = torch.stack(_random_clips([(120, 160)] * 2, 32, 3, 53)).cuda()
    with torch.no_grad():
        y = model.forward_frames(fr, crop_size=S, spatial_idx=views).cpu()
        plans = list(model._plans.values())
        y_list = model.forward_frames(list(fr), crop_size=S, spatial_idx=views).cpu()
    assert list(model._plans.values()) == plans
    assert torch.equal(y, y_list)


@pytest.mark.parametrize("name,frames,precision", [
    ("slowfast_r50", 32, "fp16"), ("shufflenetv2_w05", 16, "fp16"), ("slow_r50", 8, "fp16"),
    ("slowfast_r50", 32, "fp32")])
def test_forward_frames_clip_list_equals_forward_on_oracle_clips(esf_lib, name, frames, precision):
    cfg, model, _ = helpers.case_model_and_weights(name, precision)
    model = model.cuda().eval()
    S, views = 112, (0, 1, 2)
    clips = _random_clips(SMALL[:4], frames, 3, 54)
    single = model.num_pathways == 1
    xs = _oracle(clips, cfg.DATA.MEAN, cfg.DATA.STD, 1 if single else cfg.SLOWFAST.ALPHA, S, views, single)
    dev = [c.cuda() for c in clips]
    with torch.no_grad():
        y_ref = model([t.cuda() for t in xs]).cpu()
        y = model.forward_frames(dev, crop_size=S, spatial_idx=views).cpu()
        y2 = model.forward_frames(tuple(dev), crop_size=S, spatial_idx=list(views)).cpu()     # graph replay
    assert y.shape[0] == 12 and torch.isfinite(y).all()
    assert torch.equal(y, y_ref)
    assert torch.equal(y, y2)


def test_mixed_batches_of_one_size_share_one_plan(esf_lib):
    _, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    S, views = 112, (0, 1, 2)
    with torch.no_grad():
        model.forward_frames([c.cuda() for c in _random_clips(SMALL[:3], 32, 3, 55)], crop_size=S, spatial_idx=views)
        plans = list(model._plans.values())
        assert len(plans) == 1
        for sizes in (SMALL[2:], [(224, 112), (112, 300), (113, 129)]):
            model.forward_frames([c.cuda() for c in _random_clips(sizes, 32, 3, 56)], crop_size=S, spatial_idx=views)
            assert list(model._plans.values()) == plans


def test_clipstream_clip_lists_equal_forward_frames(esf_lib):
    import efficient_slowfast_b200 as esf

    _, model, _ = helpers.case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    S, views = 112, (0, 1, 2)
    st = esf.ClipStream(model, [(3, 32, 160, 160, 3)], frames=True, crop_size=S, spatial_idx=views)
    too_many_bytes = [c.pin_memory() for c in _random_clips([(160, 200)] * 3, 32, 3, 57)]
    too_many_clips = [c.pin_memory() for c in _random_clips([(112, 112)] * 4, 32, 3, 58)]
    for bad in (too_many_bytes, too_many_clips):
        with pytest.raises(rt.EsfError):
            st.submit(bad)
    sizes = [SMALL[:3], SMALL[2:5], [SMALL[4], SMALL[0], SMALL[1]], SMALL[3:5]]     # the last batch is short
    batches = [[c.pin_memory() for c in _random_clips(sz, 32, 3, 60 + i)] for i, sz in enumerate(sizes)]
    got = []
    with torch.no_grad():
        for b in batches:
            r = st.submit(b)
            if r is not None:
                got.append(r)
        got += st.flush()
        want = [model.forward_frames([c.cuda() for c in b], crop_size=S, spatial_idx=views).cpu() for b in batches]
    assert [i for i, _ in got] == [0, 1, 2, 3]
    for (_, y), w, b in zip(got, want, batches):
        assert y.shape[0] == 3 * len(b)
        assert torch.equal(y, w)
