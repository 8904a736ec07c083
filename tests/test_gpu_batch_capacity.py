"""Batch capacity (cfg.ESF.MAX_BATCH): one plan family per per-clip input shape.  A variant compiled at b <= N rows
reuses the capacity plan's memory and weights and must give, bit for bit, what a dedicated plan of b rows (MAX_BATCH
off) gives, on every entry point."""
import functools
import gc

import pytest
import torch

import helpers
from efficient_slowfast_b200 import engine, engine_fp32, nets_efficient, nets_resnet
from efficient_slowfast_b200 import runtime as rt

pytestmark = pytest.mark.gpu

N = 4
# host-side weight preparation: none of these may run while a variant is compiled
PREP = [(nets_resnet, "fold_conv_bn"), (nets_efficient, "fold_conv_bn"), (engine, "fold_conv_bn"),
        (engine_fp32, "fold_conv_bn"), (engine, "host64"), (engine, "bn_affine"), (engine, "attention_projection"),
        (engine, "conv_weight_bias"), (engine, "nonlocal_offset"), (engine, "pack_igemm_weight"),
        (engine, "pack_wfold_band"), (engine, "pack_stem_band"), (engine, "pack_stem_tband"), (engine, "to_device"),
        (engine_fp32, "split_weight_rows"), (engine_fp32, "split_operand_weight"), (engine.Plan, "_upload")]


def _models(name, n, precision="fp16", build=None):
    """(cfg, dedicated model, family model with MAX_BATCH = n) on the GPU, same weights."""
    cfg, model, _ = build(name, precision) if build else helpers.case_model_and_weights(name, precision)
    cfg.ESF.MAX_BATCH = n
    fam = model.__class__(cfg)
    fam.load_state_dict(model.state_dict())
    return cfg, model.cuda().eval(), fam.cuda().eval()


def _batch(name, tag, n):
    """n clips: the golden's clips, then the same clips mirrored along W (the slow clip stays the fast one's subset)."""
    xs = helpers.case_inputs(name, tag)
    out = [torch.cat([x, x.flip(-1)]) for x in xs]
    while out[0].shape[0] < n:
        out = [torch.cat([x, x.roll(7, -2)]) for x in out]
    return [x[:n].contiguous() for x in out]


def _counting(monkeypatch):
    calls = {}
    for mod, attr in PREP:
        fn = getattr(mod, attr)

        def counted(*a, _fn=fn, _key="%s.%s" % (getattr(mod, "__name__", mod), attr), **k):
            calls[_key] = calls.get(_key, 0) + 1
            return _fn(*a, **k)

        monkeypatch.setattr(mod, attr, functools.wraps(fn)(counted))
    return calls


def _rows(xs, b):
    return [x[:b].contiguous().cuda() for x in xs]


@pytest.mark.parametrize("name,tag,precision", [
    ("slowfast_r50", "s64", "fp16"), ("dual_r50", "s64", "fp16"), ("shufflenetv2_w05", "s112", "fp16"),
    ("ghostnet_w1", "s64", "fp16"), ("slow_nln_r50", "s64", "fp16"), ("dual_r50", "s64", "fp32")])
def test_variants_equal_dedicated_plans(esf_lib, monkeypatch, name, tag, precision):
    """b in {1, 2, N-1, N}: the variant's output equals a dedicated plan's; building a variant folds and packs
    nothing and adds almost no device memory; the family is one plan of the LRU."""
    _, model, fam = _models(name, N, precision)
    xs = _batch(name, tag, N)
    calls = _counting(monkeypatch)
    got = {}
    with torch.no_grad():
        got[N] = fam(_rows(xs, N)).cpu()                  # the capacity plan
        assert sum(calls.values()) > 0
        prep = dict(calls)
        cap = next(iter(fam._plans.values()))[1]
        gc.collect()                                      # plans of earlier tests are freed now, not in the window
        torch.cuda.synchronize()
        mem = torch.cuda.memory_allocated()
        for b in (1, 2, N - 1):
            got[b] = fam(_rows(xs, b)).cpu()
        gc.collect()
        torch.cuda.synchronize()
        grown = torch.cuda.memory_allocated() - mem
        assert calls == prep, "a variant ran host weight preparation: %s" % {
            k: v - prep.get(k, 0) for k, v in calls.items() if v != prep.get(k, 0)}
        assert len(fam._plans) == 1 and sorted(cap.variants) == [1, 2, N - 1]
        assert grown < 0.01 * cap.arena_bytes(), (grown, cap.arena_bytes())
        again = fam(_rows(xs, 1)).cpu()                   # after the capacity plan ran again
        fam(_rows(xs, N))
        assert torch.equal(fam(_rows(xs, 1)).cpu(), again)
        for b in (1, 2, N - 1, N):
            want = model(_rows(xs, b)).cpu()
            assert torch.isfinite(want).all()
            assert torch.equal(got[b], want), "b = %d" % b
        assert torch.equal(again, got[1])
    print("%s %s: capacity arena %.1f MB, variants added %.3f MB" % (name, precision, cap.arena_bytes() / 2 ** 20,
                                                                     grown / 2 ** 20))


def test_every_batch_size_shares_one_arena(esf_lib):
    """b = 1 .. N on slowfast_r50: one entry in the plan LRU, one set of buffers."""
    _, _, fam = _models("slowfast_r50", N)
    xs = _batch("slowfast_r50", "s64", N)
    with torch.no_grad():
        for b in range(1, N + 1):
            fam(_rows(xs, b))
            assert len(fam._plans) == 1
        cap = next(iter(fam._plans.values()))[1]
        for b, v in cap.variants.items():
            assert v.arena_bytes() == cap.arena_bytes()       # every storage a variant keeps is the capacity plan's
            for own, big in zip(v.inputs, cap.inputs):
                assert own.data_ptr() == big.data_ptr() and own.shape[0] == b
        bufs = fam.input_buffers([tuple(x[:2].shape) for x in xs])
        assert [t.data_ptr() for t in bufs] == [t.data_ptr() for t in cap.inputs]
        for t, x in zip(bufs, xs):
            t.copy_(x[:2])
        assert torch.equal(fam(bufs).cpu(), fam(_rows(xs, 2)).cpu())


def test_refusals_and_weight_edit(esf_lib):
    """b > N raises EsfError before a plan is compiled or a kernel launched; a weight edit drops the whole family."""
    _, model, fam = _models("slowfast_r50", N)
    xs = _batch("slowfast_r50", "s64", N)
    big = [torch.cat([x, x[:1]]).cuda() for x in xs]
    with torch.no_grad():
        with pytest.raises(rt.EsfError):
            fam(big)
        assert len(fam._plans) == 0
        fam(_rows(xs, 2))
        cap = next(iter(fam._plans.values()))[1]
        with pytest.raises(rt.EsfError):
            fam.forward_fast(big[1])
        with pytest.raises(rt.EsfError):
            fam.input_buffers([tuple(x.shape) for x in big])
        assert next(iter(fam._plans.values()))[1] is cap and sorted(cap.variants) == [2]
        for m in (model, fam):
            m.head.projection.weight.mul_(1.5)              # versioned in-place edit
        y = fam(_rows(xs, 2)).cpu()
        assert len(fam._plans) == 1
        new = next(iter(fam._plans.values()))[1]
        assert new is not cap and sorted(new.variants) == [2]
        assert torch.equal(y, model(_rows(xs, 2)).cpu())


def test_detection_variants(esf_lib):
    """AVA head: the variant's box rows equal a dedicated plan's, with the detection rows shared by the family."""
    from test_gpu_detection import _boxes, _clip, _detection_model

    cfg, model, fam = _models("slowfast_r50", N, build=lambda n, p: _detection_model(n, p) + (None,))
    xs = _clip(cfg, N, 64, 96)
    with torch.no_grad():
        for b in (N, 1, 2, N - 1):
            boxes = _boxes(5 + 3 * b, b, 64, 96, seed=b)
            y = fam(_rows(xs, b), boxes).cpu()
            assert torch.equal(y, model(_rows(xs, b), boxes).cpu()), "b = %d" % b
            assert torch.equal(fam.forward_fast(xs[1][:b].contiguous().cuda(), boxes).cpu(), y)
        assert len(fam._plans) == 1


def _frames(n, T, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n, T, H, W, 3), generator=g, dtype=torch.uint8)


def test_entry_points(esf_lib):
    """forward_frames (crops, ragged list, frame_index, plain), forward_fast, forward_videos with 1, 2, 3 videos and
    ClipStream video mode over batches of 3, 1, 2 videos, on one family of 3 x num_clips x V rows."""
    import efficient_slowfast_b200 as esf

    nc, views, S = 2, (0, 1, 2), 64
    rows = 3 * nc * len(views)
    cfg, model, fam = _models("slowfast_r50", rows)
    T = int(cfg.DATA.NUM_FRAMES)
    vids = [_frames(1, 40 + 9 * i, 72 + 8 * i, 96, 30 + i)[0] for i in range(3)]
    with torch.no_grad():
        def same(call):
            want = call(model).cpu()
            assert torch.equal(call(fam).cpu(), want)
            return want

        for nv in (1, 2, 3):
            same(lambda m: m.forward_videos([v.cuda() for v in vids[:nv]], fps=25.0, num_clips=nc, crop_size=S,
                                            spatial_idx=views))
        fr = _frames(2, T, 72, 96, 5).cuda()
        same(lambda m: m.forward_frames(fr, crop_size=S, spatial_idx=views))
        same(lambda m: m.forward_frames(fr[:1], crop_size=S, spatial_idx=(1,)))
        clips = [_frames(1, T, 64 + 16 * i, 80, 9 + i)[0].cuda() for i in range(3)]
        same(lambda m: m.forward_frames(clips, crop_size=S, spatial_idx=(0, 2)))
        plain = _frames(5, T, S, S, 11).cuda()
        same(lambda m: m.forward_frames(plain))
        idx = [torch.tensor(ix, dtype=torch.int32).cuda() for ix in (range(0, T, T // 4), range(T))]
        same(lambda m: m.forward_frames(plain[:3], frame_index=idx))
        fast = torch.randn(2, 3, T, S, S).cuda()
        same(lambda m: m.forward_fast(fast))
        assert len(fam._plans) == 1                          # one per-clip shape: every route above shares the family

        st = esf.ClipStream(fam, [(3, 60, 88, 96, 3)], frames=True, num_clips=nc, crop_size=S, spatial_idx=views)
        batches = [[v.pin_memory() for v in vids[:n]] for n in (3, 1, 2)]
        got = []
        for bt in batches:
            out = st.submit(bt, fps=25.0)
            if out is not None:
                got.append(out)
        got += st.flush()
        assert [i for i, _ in got] == [0, 1, 2]
        for (_, y), bt in zip(got, batches):
            want = model.forward_videos([v.cuda() for v in bt], fps=25.0, num_clips=nc, crop_size=S, spatial_idx=views)
            assert torch.equal(y, want.cpu())
        assert len(fam._plans) == 1
