"""The FP32-accurate plan (cfg.ESF.PRECISION = "fp32") across the whole ResNet family: the fully-convolutional test head,
grouped bottlenecks (RESNET.NUM_GROUPS > 1), Non-local blocks with temporal groups (NONLOCAL.GROUP > 1) and attention head
dims outside {8, 16, 32, 64, 128}.

Model tests compare with the reference's FP32 goldens where they exist, else with the CPU oracle evaluated in FP64 on the
same seeded weights and clip; piece tests compare with torch FP64 math on the same FP32 operands."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import helpers
import spatial_oracle as SO
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.build import build_model
from efficient_slowfast_b200.engine_fp32 import PrecisePlan
from efficient_slowfast_b200.workloads import pack_pathway_output, seeded_clip, seeded_state_dict
from oracle import slowfast_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FP32_TOL = 1e-4


def _ncdhw(t):
    return t.permute(0, 4, 1, 2, 3).contiguous()


def _run(model, xs):
    with torch.no_grad():
        y = model([t.cuda() for t in xs]).cpu()
        y2 = model([t.cuda() for t in xs]).cpu()      # CUDA-graph replay
    torch.cuda.synchronize()
    return y, y2


# ------------------------------------------------------------------------------------------------ goldens
@pytest.mark.parametrize("name,tag,tol", [
    ("slowfast_r50_fcn", "s96", FP32_TOL),    # head pool [4,2,2] / [32,2,2] on a 3 x 3 map: 2 x 2 positions
    ("slowfast_r50_fcn", "s64", FP32_TOL),    # the same model with the head pool covering the map
    ("dual_r18_gray", "s128", FP32_TOL),      # the fork's product config at its TEST_CROP_SIZE: 2 x 2 positions
    # RESNET.NUM_GROUPS 2, measured 1.02e-4.  The golden is 2.2e-6 from the FP64 oracle, so the error is this plan's: the
    # tensor core's FP32 accumulator rounds toward zero once per MMA (~1e-9 per product, test_conv_fp32_path).  Scaling
    # every conv output of the FP64 oracle by (1 - 1e-9 K) moves the probabilities of slowfast_r50 s64 by 3.5e-5 (this
    # plan: 4.1e-5) and those of this draw by 8.8e-5 with K of one group, 1.2e-4 with the block-diagonal layer's full K:
    # the g2 draw amplifies the same rounding 2.5x more, and the fold adds up to 1.35x.  1.5e-4 is written for it.
    ("slowfast_r50_g2", "s64", 1.5e-4)])
def test_fp32_family_matches_reference_golden(esf_lib, name, tag, tol):
    xs = helpers.case_inputs(name, tag)
    _, model, gold = helpers.case_model_and_weights(name, "fp32")
    y, y2 = _run(model.cuda().eval(), xs)
    _, model16, _ = helpers.case_model_and_weights(name, "fp16")
    y16, _ = _run(model16.cuda().eval(), xs)
    ref = torch.as_tensor(gold[tag + "/probs"])
    err, err16 = helpers.rel_err(y, ref), helpers.rel_err(y16, ref)
    print("%s/%s: rel err of probs fp32 %.3e, fp16 %.3e (tol %.1e)" % (name, tag, err, err16, tol))
    assert err <= tol
    assert err < err16
    assert torch.equal(y.argmax(1), ref.argmax(1))
    assert torch.equal(y, y2)
    assert abs(y.sum(1) - 1).max() < 1e-5


# ------------------------------------------------------------------------------------------------ CPU oracle in FP64
def _oracle_case(cfg, bn_stats, inputs):
    """FP32 plan and FP64 oracle on the recipe's seeded weights (BN statistics from a golden when its shapes match, else
    the identity statistics) -> (fp32 probs, fp64 probs, plan)."""
    cfg.ESF.PRECISION = "fp32"
    torch.manual_seed(0)
    model = build_model(cfg)
    model.load_state_dict(seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn_stats), strict=True)
    model = model.cuda().eval()
    y, y2 = _run(model, inputs)
    assert torch.equal(y, y2)
    yo = O.forward(cfg, {k: v.cpu() for k, v in model.state_dict().items()}, inputs, dtype=torch.float64)
    plan = next(reversed(model._plans.values()))[1]
    return y, yo.cpu(), plan


def test_fp32_nonlocal_group2_matches_fp64_oracle(esf_lib):
    """Slow 8x8 R50 with Non-local blocks after res3 blocks 1,3 and res4 blocks 1,3,5, NONLOCAL.GROUP 2 (the blocks see
    two 4-frame halves of every clip).  Weights and BN statistics are those of the slow_nln_r50 golden: the group is a
    reshaping only, the parameter shapes are the same.  The Non-local blocks of this draw amplify every perturbation
    (test_gpu_fp32_path: 1.8e-4 against the reference's FP32 forward), so the bound is twice the GROUP 1 figure of the
    same weights and clip."""
    gold = helpers.load_golden("slow_nln_r50")
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    xs = helpers.case_inputs("slow_nln_r50", "s64")
    errs = {}
    for group in (1, 2):
        cfg = helpers.case_cfg("slow_nln_r50")
        cfg.NONLOCAL.GROUP = [[group if loc else 1] for loc, in cfg.NONLOCAL.LOCATION]
        y, yo, plan = _oracle_case(cfg, bn, xs)
        errs[group] = helpers.rel_err(y, yo)
        assert torch.equal(y.argmax(1), yo.argmax(1))
        if group == 2:
            assert any("N=%dx" % (4 * 8 * 8) in m["label"] for m in plan.meta if m["kind"] == "nl_gemm")
    print("slow_nln_r50 s64 vs FP64 oracle: GROUP 1 %.3e, GROUP 2 %.3e" % (errs[1], errs[2]))
    assert errs[2] <= 2 * errs[1]


def test_fp32_attention_head_dim_4_matches_fp64_oracle(esf_lib):
    """SlowFastDualAttention R50 with WIDTH_PER_GROUP 32: the s1 fuse attends with head dim 32 / BETA_INV = 4 (then 16,
    32, 64).  No golden and no calibrated BN statistics exist for this width: identity statistics, FP64 oracle."""
    cfg = helpers.case_cfg("dual_r50")
    cfg.RESNET.WIDTH_PER_GROUP = 32
    xs = pack_pathway_output(seeded_clip(2, 32, 64, seed=1), cfg.SLOWFAST.ALPHA)
    y, yo, plan = _oracle_case(cfg, None, xs)
    dims = sorted({int(m["label"].split("d=")[1].split()[0]) for m in plan.meta if m["kind"] == "attention"})
    err = helpers.rel_err(y, yo)
    print("dual R50 width 32 (head dims %s) vs FP64 oracle: rel err %.3e" % (dims, err))
    assert dims == [4, 16, 32, 64]
    assert err <= FP32_TOL
    assert torch.equal(y.argmax(1), yo.argmax(1))


# ------------------------------------------------------------------------------------------------ pieces
@pytest.mark.parametrize("act", [rt.HEAD_SOFTMAX, rt.HEAD_SIGMOID])
def test_fp32_head_positions(esf_lib, act):
    """PrecisePlan.head_positions (AvgPool3d stride 1 -> Linear -> softmax / sigmoid at every position -> mean) vs torch
    FP64 on the same FP32 activations, two pathways sliced out of wider buffers."""
    g = torch.Generator().manual_seed(11 + act)
    B, K = 3, 400
    plan = PrecisePlan(DEV)
    xs = []
    for (T, H, W, C), off in (((4, 3, 3, 64), 8), ((32, 3, 3, 8), 0)):
        buf = plan.act(B, T, H, W, C + 8)
        buf.f32.copy_(torch.randn(buf.f32.shape, generator=g).to(DEV))
        xs.append(buf[..., off:off + C])
    pools = [(4, 2, 2), (32, 2, 2)]
    w = torch.randn(K, 72, generator=g) * 0.3
    b = torch.randn(K, generator=g) * 0.1
    out = plan.head_positions(xs, pools, w, b, act)
    plan.launch_all()
    torch.cuda.synchronize()
    pooled = [F.avg_pool3d(_ncdhw(x.f32).double().cpu(), ps, stride=1) for x, ps in zip(xs, pools)]
    z = F.linear(torch.cat(pooled, 1).permute(0, 2, 3, 4, 1), w.double(), b.double())
    ref = (torch.softmax(z, -1) if act == rt.HEAD_SOFTMAX else torch.sigmoid(z)).mean((1, 2, 3))
    err = helpers.rel_err(out.cpu(), ref)
    print("fp32 head at 2x2 positions (act %d): rel err %.3e" % (act, err))
    assert err <= 1e-6


@pytest.mark.parametrize("groups,cin,cout,k,pad", [(2, 64, 64, (1, 3, 3), (0, 1, 1)), (4, 128, 128, (1, 3, 3), (0, 1, 1)),
                                                   (2, 32, 64, (3, 1, 1), (1, 0, 0)), (32, 256, 256, (1, 3, 3), (0, 1, 1))])
def test_grouped_conv_fp32_path(esf_lib, groups, cin, cout, k, pad):
    """Grouped split-operand convolution (one GEMM over the block-diagonal weight) vs torch FP64 grouped conv3d of the same
    FP32 operands; bound of test_conv_fp32_path with K = the dense reduction length."""
    g = torch.Generator().manual_seed(groups + cin)
    B, T, H, W = 2, 4, 14, 14
    plan = PrecisePlan(DEV)
    xbuf = plan.act(B, T, H, W, cin + 16)
    xbuf.f32.copy_((torch.randn(xbuf.f32.shape, generator=g) * 2).to(DEV))
    plan._post(xbuf.f32, xbuf, label="split")
    x = xbuf[..., 16:]
    y = plan.act(B, T, H, W, cout)
    w = torch.randn(cout, cin // groups, *k, generator=g).double() * (2.0 / (cout * k[0] * k[1] * k[2])) ** 0.5
    bias = torch.randn(cout, generator=g).double() * 0.1
    plan.conv(x, y, w, bias, padding=pad, groups=groups, act=rt.ACT_RELU)
    plan.launch_all()
    torch.cuda.synchronize()
    ref = F.conv3d(_ncdhw(x.f32).double().cpu(), w, bias, padding=pad, groups=groups).relu()
    err = helpers.rel_err(_ncdhw(y.f32).cpu(), ref)
    K = 3 * cin * k[0] * k[1] * k[2]
    print("grouped conv g%d %d->%d %s: rel err %.3e" % (groups, cin, cout, k, err))
    assert err <= 4e-9 * K + 1e-6
    assert sum(m["kind"] == "conv_igemm" for m in plan.meta) == 1


def test_depthwise_conv_is_not_part_of_fp32_plan(esf_lib):
    plan = PrecisePlan(DEV)
    x, y = plan.act(1, 2, 8, 8, 16), plan.act(1, 2, 8, 8, 16)
    with pytest.raises(NotImplementedError):
        plan.conv(x, y, torch.zeros(16, 1, 1, 3, 3, dtype=torch.float64), torch.zeros(16, dtype=torch.float64),
                  padding=(0, 1, 1), groups=16)


def _attention_case(d, T, H, W, alpha, seed):
    g = torch.Generator().manual_seed(seed)
    B, N = 2, T * H * W
    proj = torch.randn(B, N, 4 * d, generator=g)
    proj[:, :, d:3 * d] *= (6.0 / d) ** 0.5
    scale, shift = torch.rand(d, generator=g) + 0.5, torch.randn(d, generator=g) * 0.2
    gamma = 0.7
    p = proj.double().reshape(B, N, 4, d)
    att = torch.softmax(p[:, :, 1] @ p[:, :, 2].transpose(1, 2), dim=-1)
    ref = ((gamma * (att @ p[:, :, 3]) + p[:, :, 0]) * scale.double() + shift.double()).relu()
    ref = ref.reshape(B, T, H, W, d).repeat_interleave(alpha, dim=1)
    ybuf = torch.full((B, T * alpha, H, W, d + 16), 7.0, dtype=torch.float32, device=DEV)
    return proj.to(DEV), scale.to(DEV), shift.to(DEV), gamma, ref, ybuf


@pytest.mark.parametrize("d,T,H,W,alpha", [(4, 2, 9, 7, 4), (12, 4, 12, 10, 4), (24, 2, 14, 14, 2), (40, 2, 7, 7, 2)])
def test_attention_split_tensor_core_padded_head_dims(esf_lib, d, T, H, W, alpha):
    """esf_attn_tc_create_split at head dims its geometry pads (Q~/K~ rows, V^T and V_lo^T rows beyond d) vs FP64; the
    neighbours of the output slice stay untouched."""
    L = esf_lib
    pj, sc, sh, gamma, ref, ybuf = _attention_case(d, T, H, W, alpha, d + T + H)
    B, N = 2, T * H * W
    y = ybuf[..., 8:8 + d]
    packed = torch.empty(L.esf_attn_tc_pack_bytes(B, N, d), dtype=torch.uint8, device=DEV)
    vlo = torch.empty(L.esf_attn_tc_vlo_bytes(B, N, d), dtype=torch.uint8, device=DEV)
    yv = rt.view(y)
    h = ctypes.c_void_p()
    rt.check(L.esf_attn_tc_pack(pj.data_ptr(), B, N, d, rt.F16, packed.data_ptr(), None))
    rt.check(L.esf_attn_tc_pack_vlo(pj.data_ptr(), B, N, d, vlo.data_ptr(), None))
    rt.check(L.esf_attn_tc_create_split(packed.data_ptr(), vlo.data_ptr(), B, T, H, W, d, gamma, sc.data_ptr(),
                                        sh.data_ptr(), alpha, ctypes.byref(yv), ctypes.byref(h)))
    rt.check(L.esf_op_launch(h, None))
    torch.cuda.synchronize()
    L.esf_op_destroy(h)
    err = helpers.rel_err(y.cpu(), ref)
    print("split tcgen05 attention d=%d N=%d: rel err %.3e" % (d, N, err))
    assert err <= 2e-5
    assert (ybuf[..., :8] == 7.0).all() and (ybuf[..., 8 + d:] == 7.0).all()


@pytest.mark.parametrize("d,T,H,W,alpha", [(72, 2, 7, 7, 2), (90, 1, 9, 8, 4), (100, 2, 5, 7, 1), (5, 2, 9, 7, 4)])
def test_attention_fp32_any_head_dim(esf_lib, d, T, H, W, alpha):
    """esf_p32_attention at head dims below its compiled widths (scalar loads when d % 4 != 0) vs FP64."""
    pj, sc, sh, gamma, ref, ybuf = _attention_case(d, T, H, W, alpha, d + T)
    y = ybuf[..., 8:8 + d]
    yv = rt.view(y)
    rt.check(esf_lib.esf_p32_attention(pj.data_ptr(), 2, T, H, W, d, gamma, sc.data_ptr(), sh.data_ptr(), alpha,
                                       ctypes.byref(yv), None), "esf_p32_attention")
    torch.cuda.synchronize()
    err = helpers.rel_err(y.cpu(), ref)
    print("p32 attention d=%d: rel err %.3e" % (d, err))
    assert err <= 5e-6
    assert (ybuf[..., :8] == 7.0).all() and (ybuf[..., 8 + d:] == 7.0).all()


def test_attention_generic_fp32_output(esf_lib):
    """esf_attn_generic into an FP32 slice (the FP32-accurate plan above d = 128) vs FP64."""
    d, T, H, W, alpha = 144, 2, 7, 7, 2
    pj, sc, sh, gamma, ref, ybuf = _attention_case(d, T, H, W, alpha, 5)
    y = ybuf[..., 8:8 + d]
    yv = rt.view(y)
    rt.check(esf_lib.esf_attn_generic(pj.data_ptr(), 2, T, H, W, d, gamma, sc.data_ptr(), sh.data_ptr(), alpha,
                                      ctypes.byref(yv), None), "esf_attn_generic")
    torch.cuda.synchronize()
    err = helpers.rel_err(y.cpu(), ref)
    print("generic attention d=%d, FP32 out: rel err %.3e" % (d, err))
    assert err <= 5e-6
    assert (ybuf[..., :8] == 7.0).all() and (ybuf[..., 8 + d:] == 7.0).all()


# ------------------------------------------------------------------------------------------------ test protocol
def test_fp32_fcn_test_protocol_end_to_end(esf_lib):
    """The reference's test protocol in the FP32 plan: decode-size uint8 frames, short side resized to the test crop,
    three uniform crops, fully-convolutional head.  forward_frames and ClipStream give exactly forward() on the test
    loader oracle's clips."""
    import efficient_slowfast_b200 as esf

    cfg, model, _ = helpers.case_model_and_weights("slowfast_r50_fcn", "fp32")
    model = model.cuda().eval()
    S, views = 96, (0, 1, 2)
    g = torch.Generator().manual_seed(42)
    batches = [torch.randint(0, 256, (1, 32, 120, 160, 3), generator=g, dtype=torch.uint8).pin_memory()
               for _ in range(2)]
    st = esf.ClipStream(model, [tuple(batches[0].shape)], frames=True, crop_size=S, spatial_idx=views)
    got = []
    with torch.no_grad():
        for b in batches:
            r = st.submit([b])
            if r is not None:
                got.append(r)
        got += st.flush()
        for (i, ys), fr in zip(got, batches):
            xs = SO.frames_to_crop_inputs(fr, cfg.DATA.MEAN, cfg.DATA.STD, cfg.SLOWFAST.ALPHA, S, views)
            want = model([t.cuda() for t in xs]).cpu()
            yf = model.forward_frames(fr.cuda(), crop_size=S, spatial_idx=views).cpu()
            assert want.shape[0] == 3 and abs(want.sum(1) - 1).max() < 1e-5
            assert torch.equal(yf, want)
            assert torch.equal(ys, want)
    assert [i for i, _ in got] == [0, 1]
