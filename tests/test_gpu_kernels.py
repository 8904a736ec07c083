"""GPU parity of every kernel behind the C ABI against plain torch FP32/FP64 math on the same (BF16-rounded)
operands.  Tolerances are stated per test; BF16 outputs carry 2^-9 relative rounding."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.engine import Plan, stem_route

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand_act(g, B, T, H, W, C, scale=1.0, dtype=torch.bfloat16):
    return (torch.randn(B, T, H, W, C, generator=g) * scale).to(dtype)


def _to_ncdhw(t):
    return t.float().permute(0, 4, 1, 2, 3).contiguous()


def _to_ndhwc(t):
    return t.permute(0, 2, 3, 4, 1).contiguous()


def _diagnose(name, got, ref, thr):
    """Print where a conv result is wrong (which channels / positions), to debug without a local GPU."""
    bad = (got - ref).abs() > thr
    print("DIAG %s: %d / %d elements wrong; got finite %s; got==7 fraction %.3f; got==0 fraction %.3f" % (
        name, int(bad.sum()), bad.numel(), bool(torch.isfinite(got).all()), float((got == 7).float().mean()),
        float((got == 0).float().mean())))
    B, C, T, H, W = got.shape
    per_c = bad.float().mean((0, 2, 3, 4))
    print("DIAG wrong fraction per channel (first 32):", [round(float(v), 2) for v in per_c[:32]])
    print("DIAG wrong fraction per 8-channel chunk:", [round(float(v), 2) for v in per_c.reshape(-1, 8).mean(1)[:32]])
    print("DIAG wrong fraction per t:", [round(float(v), 2) for v in bad.float().mean((0, 1, 3, 4))])
    print("DIAG wrong fraction per h:", [round(float(v), 2) for v in bad.float().mean((0, 1, 2, 4))])
    print("DIAG wrong fraction per w:", [round(float(v), 2) for v in bad.float().mean((0, 1, 2, 3))])
    print("DIAG wrong fraction per b:", [round(float(v), 2) for v in bad.float().mean((1, 2, 3, 4))])
    idx = bad.nonzero()[:6]
    for i in idx:
        i = tuple(int(v) for v in i)
        print("DIAG  at (b,c,t,h,w)=%s got %.4f ref %.4f" % (i, float(got[i]), float(ref[i])))
    print("DIAG got[0,:8,0,0,0] ", got[0, :8, 0, 0, 0].tolist())
    print("DIAG ref[0,:8,0,0,0] ", ref[0, :8, 0, 0, 0].tolist())


CONV_CASES = [
    # name, (B,T,H,W), Cin, Cout, kernel, stride, pad, dil, act, res, out_f32
    ("plain_1x1_one_tile", (1, 1, 8, 16), 64, 64, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 0, False, False),
    ("plain_1x1_k128", (1, 2, 8, 16), 128, 128, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 0, False, False),
    ("c_1x1_res_relu", (2, 4, 14, 14), 64, 256, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 1, True, False),
    ("a_3x1x1_2chunks", (2, 8, 7, 7), 128, 32, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1), 1, False, False),
    ("b_1x3x3", (1, 2, 28, 28), 64, 64, (1, 3, 3), (1, 1, 1), (0, 1, 1), (1, 1, 1), 1, False, False),
    ("b_1x3x3_s2_kc16", (2, 4, 28, 28), 16, 16, (1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 1), 1, False, False),
    ("proj_1x1_s2_partial_chunk", (1, 2, 56, 56), 72, 128, (1, 1, 1), (1, 2, 2), (0, 0, 0), (1, 1, 1), 0, False, False),
    ("b_1x3x3_kc32", (2, 4, 14, 14), 32, 32, (1, 3, 3), (1, 1, 1), (0, 1, 1), (1, 1, 1), 1, False, False),
    ("lateral_5x1x1_s8", (2, 32, 14, 14), 8, 16, (5, 1, 1), (8, 1, 1), (2, 0, 0), (1, 1, 1), 1, False, False),
    ("lateral_7x1x1_s4", (1, 32, 7, 7), 32, 64, (7, 1, 1), (4, 1, 1), (3, 0, 0), (1, 1, 1), 1, False, False),
    ("proj_f32_out", (2, 2, 14, 14), 256, 128, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 0, False, True),
    ("proj_f32_out_n32", (2, 2, 14, 14), 64, 32, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 0, False, True),
    ("wide_2048", (4, 2, 7, 7), 512, 2048, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 1, True, False),
    ("b_1x3x3_dil2", (1, 2, 14, 14), 64, 64, (1, 3, 3), (1, 1, 1), (0, 2, 2), (1, 2, 2), 1, False, False),
    ("tiny_8to32", (2, 8, 14, 14), 8, 32, (1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1), 0, True, False),
    ("b_1x3x3_s2_7x7", (3, 8, 14, 14), 512, 512, (1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 1), 1, False, False),
    ("many_tiles", (8, 8, 28, 28), 128, 128, (1, 3, 3), (1, 1, 1), (0, 1, 1), (1, 1, 1), 1, False, False),
    # k x 1 x 1, stride 1: residual over two K chunks, T not a multiple of the box, odd sizes, FP32 output
    ("t3x1x1_64to16", (2, 32, 28, 28), 64, 16, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1), 1, False, False),
    ("t3x1x1_res_2chunks", (1, 16, 14, 14), 128, 32, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1), 1, True, False),
    ("t5x1x1_partial_t", (1, 13, 8, 16), 64, 64, (5, 1, 1), (1, 1, 1), (2, 0, 0), (1, 1, 1), 0, False, False),
    ("t3x1x1_kc32_odd", (2, 9, 7, 9), 32, 16, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1), 1, False, False),
    ("t3x1x1_f32_out", (1, 8, 8, 8), 64, 32, (3, 1, 1), (1, 1, 1), (1, 0, 0), (1, 1, 1), 0, False, True),
]


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("case", CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv_igemm(esf_lib, case, precision):
    name, (B, T, H, W), cin, cout, k, s, p, d, act, use_res, out_f32 = case
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(sum(map(ord, name)) % 1000)
    # input and output live inside wider concat buffers (channel slices) to exercise strided views
    xbuf = _rand_act(g, B, T, H, W, cin + 8, dtype=adt).to(DEV)
    x = xbuf[..., 8:8 + cin]
    w = torch.randn(cout, cin, *k, generator=g) * (2.0 / (cin * k[0] * k[1] * k[2])) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    ref = F.conv3d(_to_ncdhw(x.cpu()), w.to(adt).float(), bias, s, p, d)
    _, _, To, Ho, Wo = ref.shape
    res = None
    if use_res:
        res = _rand_act(g, B, To, Ho, Wo, cout, dtype=adt).to(DEV)
        ref = ref + _to_ncdhw(res.cpu())
    if act == 1:
        ref = ref.relu()
    plan = Plan(DEV, precision)
    odt = torch.float32 if out_f32 else adt
    ybuf = torch.full((B, To, Ho, Wo, cout + 16), 7.0, dtype=odt, device=DEV)
    y = ybuf[..., 8:8 + cout] if not out_f32 else ybuf[..., 4:4 + cout]
    plan.conv_igemm(x, y, w.double(), bias.double(), stride=s, padding=p, dilation=d, act=act, res=res)
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(y.cpu())
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    # FP32 out: accumulation order only; 16-bit out: + 2^-9 (BF16) / 2^-12 (FP16) output rounding
    tol = 2e-3 if (out_f32 or precision == "fp16") else 1e-2
    if not err <= tol * scale:
        _diagnose(name, got, ref, tol * scale)
    assert err <= tol * scale, "%s: max err %.4g vs scale %.4g" % (name, err, scale)
    # neighbours of the output slice are untouched
    lo = ybuf[..., :4].float()
    assert (lo == 7.0).all()
    assert (ybuf[..., -4:].float() == 7.0).all()


# name, (B,T,H,W), Cin, Cout, kernel, stride, padding, act, residual ("", "dense", "slice"), sliced output
WFOLD_CASES = [
    ("b_1x3x3_8", (2, 4, 56, 56), 8, 8, (1, 3, 3), (1, 1, 1), (0, 1, 1), 1, "", False),
    ("c_1x1x1_8to32_res", (2, 4, 56, 56), 8, 32, (1, 1, 1), (1, 1, 1), (0, 0, 0), 1, "dense", False),
    ("c_1x1x1_8to32_res_slice_out", (2, 4, 56, 56), 8, 32, (1, 1, 1), (1, 1, 1), (0, 0, 0), 1, "dense", True),
    ("c_res_slice", (2, 4, 28, 28), 16, 64, (1, 1, 1), (1, 1, 1), (0, 0, 0), 1, "slice", True),
    ("a_3x1x1_32to8", (2, 6, 56, 56), 32, 8, (3, 1, 1), (1, 1, 1), (1, 0, 0), 1, "", False),
    ("a_3x1x1_16to8", (1, 5, 56, 56), 16, 8, (3, 1, 1), (1, 1, 1), (1, 0, 0), 1, "", False),
    ("b_1x3x3_s2_16", (2, 4, 56, 56), 16, 16, (1, 3, 3), (1, 2, 2), (0, 1, 1), 1, "", False),
    ("branch1_s2_32to128", (2, 4, 28, 28), 32, 128, (1, 1, 1), (1, 2, 2), (0, 0, 0), 0, "", False),
    ("b_1x3x3_32_14", (3, 4, 14, 14), 32, 32, (1, 3, 3), (1, 1, 1), (0, 1, 1), 1, "", False),
    ("c_32to128_14_slice", (3, 4, 14, 14), 32, 128, (1, 1, 1), (1, 1, 1), (0, 0, 0), 1, "dense", True),
    ("odd_w_30", (1, 3, 10, 30), 8, 24, (1, 3, 3), (1, 1, 1), (0, 1, 1), 1, "dense", False),
    ("fuse_5x1x1_8to16_slice", (2, 8, 28, 28), 8, 16, (5, 1, 1), (1, 1, 1), (2, 0, 0), 1, "", True),
]


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("case", WFOLD_CASES, ids=[c[0] for c in WFOLD_CASES])
def test_conv_wfold(esf_lib, case, precision):
    """Thin layers as W-folded banded GEMMs (esf_conv_wfold_create) against torch conv3d."""
    from efficient_slowfast_b200.engine import wfold_block
    name, (B, T, H, W), cin, cout, k, s, p, act, res_kind, slice_out = case
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(sum(map(ord, name)) % 1000)
    x = _rand_act(g, B, T, H, W, cin, dtype=adt).to(DEV)
    w = torch.randn(cout, cin, *k, generator=g) * (2.0 / (cin * k[0] * k[1] * k[2])) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    ref = F.conv3d(_to_ncdhw(x.cpu()), w.to(adt).float(), bias, s, p)
    _, _, To, Ho, Wo = ref.shape
    res = None
    if res_kind:
        extra = 16 if res_kind == "slice" else 0
        rbuf = _rand_act(g, B, To, Ho, Wo, cout + extra, dtype=adt).to(DEV)
        res = rbuf[..., extra // 2:extra // 2 + cout]
        ref = ref + _to_ncdhw(res.cpu())
    if act == 1:
        ref = ref.relu()
    extra = 16 if slice_out else 0
    ybuf = torch.full((B, To, Ho, Wo, cout + extra), 7.0, dtype=adt, device=DEV)
    y = ybuf[..., extra // 2:extra // 2 + cout]
    wb = wfold_block(x, y, res, w.shape, s, p, (1, 1, 1))
    assert wb >= 2, "planner refused to fold %s" % name
    plan = Plan(DEV, precision)
    plan.conv(x, y, w.double(), bias.double(), stride=s, padding=p, act=act, res=res)
    assert plan.meta[-1]["kind"] == "conv_wfold"
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(y.cpu())
    err = (got - ref).abs().max().item()
    scale = ref.abs().max().item()
    tol = 2e-3 if precision == "fp16" else 1e-2
    if not err <= tol * scale:
        _diagnose(name, got, ref, tol * scale)
    assert err <= tol * scale, "%s (wb %d): max err %.4g vs scale %.4g" % (name, wb, err, scale)
    if slice_out:
        assert (ybuf[..., :8].float() == 7.0).all() and (ybuf[..., -8:].float() == 7.0).all()


def test_conv_direct_depthwise_and_grouped(esf_lib):
    g = torch.Generator().manual_seed(5)
    for (cin, cout, groups, k, s, p) in [(24, 24, 24, (3, 3, 3), (1, 2, 2), (1, 1, 1)),
                                         (12, 30, 3, (1, 1, 1), (1, 1, 1), (0, 0, 0)),
                                         (6, 10, 1, (1, 3, 3), (1, 1, 1), (0, 1, 1))]:
        x = _rand_act(g, 2, 4, 10, 10, cin).to(DEV)
        w = torch.randn(cout, cin // groups, *k, generator=g) * 0.2
        bias = torch.randn(cout, generator=g) * 0.1
        ref = F.conv3d(_to_ncdhw(x.cpu()), w, bias, s, p, 1, groups).relu()
        y = torch.empty(_to_ndhwc(ref).shape, dtype=torch.bfloat16, device=DEV)
        plan = Plan(DEV)
        plan.conv_direct(x, y, w.double(), bias.double(), stride=s, padding=p, groups=groups, act=rt.ACT_RELU)
        plan.launch_all()
        torch.cuda.synchronize()
        err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
        assert err <= 1e-2 * ref.abs().max().item()


@pytest.mark.parametrize("cin,cout,groups,off", [(15, 60, 3, 60), (24, 36, 1, 12), (48, 20, 1, 6)])
def test_conv_into_unaligned_concat_slice(esf_lib, cin, cout, groups, off):
    """A dense / grouped pointwise conv whose output is a concat slice at a channel offset that is not a multiple of 8
    still runs on the implicit GEMM (aligned buffer + row copy); the neighbouring channels stay untouched."""
    g = torch.Generator().manual_seed(cin + cout)
    B, T, H, W = 2, 4, 7, 7
    plan = Plan(DEV, "fp16")
    x = plan.act(B, T, H, W, cin)
    x.copy_(_rand_act(g, B, T, H, W, cin, dtype=torch.float16))
    w = torch.randn(cout, cin // groups, 1, 1, 1, generator=g) * (2.0 * groups / cin) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    ref = F.conv3d(_to_ncdhw(x.cpu()).float(), w.half().float(), bias, groups=groups).relu()
    ybuf = plan.act(B, T, H, W, off + cout + 4)
    full = next(t for t in reversed(plan.keep) if isinstance(t, torch.Tensor))
    full.fill_(7.0)
    y = ybuf[..., off:off + cout]
    plan.conv(x, y, w.double(), bias.double(), groups=groups, act=rt.ACT_RELU)
    kinds = [m["kind"] for m in plan.meta]
    assert "conv_direct" not in kinds and kinds[-1] == "shuffle", kinds
    plan.launch_all()
    torch.cuda.synchronize()
    err = (_to_ncdhw(y.cpu()).float() - ref).abs().max().item()
    assert err <= 3e-3 * ref.abs().max().item(), err
    assert (full[..., :off].float() == 7.0).all() and (full[..., off + cout:].float() == 7.0).all()


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("C,k,s,shape", [
    (144, (3, 3, 3), (1, 1, 1), (2, 4, 14, 14)), (24, (3, 3, 3), (1, 2, 2), (2, 4, 14, 14)),
    (12, (3, 3, 3), (1, 1, 1), (1, 3, 10, 9)), (18, (3, 3, 3), (1, 2, 2), (1, 3, 11, 13)),
    (27, (3, 3, 3), (1, 1, 1), (1, 2, 7, 6)), (48, (1, 3, 3), (1, 1, 1), (2, 2, 8, 8)),
    (4, (3, 3, 3), (1, 1, 1), (1, 4, 12, 12)), (320, (3, 3, 3), (1, 2, 2), (1, 2, 7, 7)),
    (40, (3, 3, 3), (2, 2, 2), (1, 4, 9, 9)), (72, (1, 5, 5), (1, 1, 1), (2, 3, 9, 9)),
    (28, (1, 5, 5), (1, 2, 2), (1, 3, 14, 14)), (7, (1, 5, 5), (1, 2, 2), (1, 2, 9, 11)),
    (12, (3, 3, 3), (1, 1, 1), (2, 10, 17, 19)),
    # marching kernel: several row segments per plane (H > 16), ragged W, stride 2 in T, weights beyond 48 KB of smem
    (144, (3, 3, 3), (1, 1, 1), (1, 3, 37, 21)), (24, (3, 3, 3), (1, 2, 2), (1, 3, 40, 23)),
    (16, (3, 3, 3), (2, 2, 2), (1, 5, 35, 35)), (8, (1, 3, 3), (1, 1, 1), (2, 2, 33, 18)),
    (960, (3, 3, 3), (1, 1, 1), (1, 2, 7, 7)), (1080, (3, 3, 3), (1, 2, 2), (1, 2, 7, 7)),
    (4, (3, 3, 3), (1, 2, 2), (1, 4, 34, 30)), (28, (3, 3, 3), (1, 1, 1), (1, 2, 18, 5))])
def test_depthwise_vector_kernel(esf_lib, C, k, s, shape, precision):
    """Depthwise convs through Plan.conv: vector kernel (VEC 8/4/2/1 by channel count), padded channel pitch, slices."""
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(C)
    B, T, H, W = shape
    plan = Plan(DEV, precision)
    x = plan.act(B, T, H, W, C)
    if C >= 8 and C % 8:
        plan.keep[-1].fill_(float("nan"))     # padding channels of the rows hold garbage in real plans
    x.copy_(_rand_act(g, B, T, H, W, C, dtype=adt))
    w = torch.randn(C, 1, *k, generator=g) * 0.3
    bias = torch.randn(C, generator=g) * 0.1
    p = (k[0] // 2, k[1] // 2, k[2] // 2)
    ref = F.conv3d(_to_ncdhw(x.cpu()), w.to(adt).float(), bias, s, p, 1, C)   # weights are held in the 16-bit format
    res = None
    if C in (12, 28, 144):      # residual fused into the depthwise epilogue (GhostNet shortcut branches)
        res = plan.act(*_to_ndhwc(ref).shape)
        res.copy_(_rand_act(g, *res.shape, dtype=adt))
        ref = ref + _to_ncdhw(res.cpu())
    ref = ref.relu()
    y = plan.act(*_to_ndhwc(ref).shape)
    plan.conv(x, y, w.double(), bias.double(), stride=s, padding=p, groups=C, act=rt.ACT_RELU, res=res)
    assert plan.meta[-1]["kind"] == "dwconv"
    # odd channel counts run over the rows' padded width with 16-byte vectors (esf_dwconv_padded)
    assert ("pad" in plan.meta[-1]["label"]) == (C >= 8 and C % 8 != 0)
    plan.launch_all()
    torch.cuda.synchronize()
    err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
    assert err <= (2e-3 if precision == "fp16" else 1e-2) * ref.abs().max().item()


@pytest.mark.parametrize("cin,cout,groups", [(27, 162, 1), (180, 1080, 1), (540, 480, 1), (240, 480, 3), (1080, 960, 3),
                                             (36, 216, 1), (120, 72, 3), (540, 480, 3), (54, 240, 3), (15, 60, 3),
                                             (120, 60, 3)])
def test_pointwise_odd_channels_on_tensor_cores(esf_lib, cin, cout, groups):
    """1x1x1 convs whose channel counts are not multiples of 8 (or are grouped) run on the implicit GEMM thanks to the
    padded channel pitch / per-group slicing; residual + ReLU fused."""
    g = torch.Generator().manual_seed(cin + cout)
    B, T, H, W = 2, 4, 7, 7
    plan = Plan(DEV, "fp16")
    x = plan.act(B, T, H, W, cin)
    x.copy_(_rand_act(g, B, T, H, W, cin, dtype=torch.float16))
    res = plan.act(B, T, H, W, cout)
    res.copy_(_rand_act(g, B, T, H, W, cout, dtype=torch.float16))
    w = torch.randn(cout, cin // groups, 1, 1, 1, generator=g) * (2.0 / (cin // groups)) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    ref = (F.conv3d(_to_ncdhw(x.cpu()), w.half().float(), bias, groups=groups) + _to_ncdhw(res.cpu())).relu()
    y = plan.act(B, T, H, W, cout)
    plan.conv(x, y, w.double(), bias.double(), groups=groups, act=rt.ACT_RELU, res=res)
    assert all(m["kind"] in ("conv_igemm", "conv_wfold") for m in plan.meta), [m["kind"] for m in plan.meta]
    assert len(plan.meta) in (1, groups)     # per-group GEMMs on aligned slices, else one block-diagonal GEMM
    plan.launch_all()
    torch.cuda.synchronize()
    err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
    assert err <= 2e-3 * ref.abs().max().item(), err


@pytest.mark.parametrize("cin,cout,use_res,slice_out", [(2, 12, False, False), (6, 36, False, False), (3, 18, False, True),
                                                        (4, 2, False, False), (18, 3, True, True), (12, 3, False, False),
                                                        (4, 24, False, False), (6, 4, True, False), (7, 7, False, False)])
def test_pointwise_tiny_channels(esf_lib, cin, cout, use_res, slice_out):
    """1x1x1 convs with C_in < 8 or C_out < 8 (first fast-pathway layers of the efficient nets): pw_small kernel."""
    g = torch.Generator().manual_seed(cin * 100 + cout)
    B, T, H, W = 2, 3, 9, 10
    plan = Plan(DEV, "fp16")
    x = plan.act(B, T, H, W, cin)
    x.copy_(_rand_act(g, B, T, H, W, cin, dtype=torch.float16))
    w = torch.randn(cout, cin, 1, 1, 1, generator=g) * (2.0 / cin) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    ref = F.conv3d(_to_ncdhw(x.cpu()), w, bias)
    res = None
    if use_res:
        res = plan.act(B, T, H, W, cout)
        res.copy_(_rand_act(g, B, T, H, W, cout, dtype=torch.float16))
        ref = ref + _to_ncdhw(res.cpu())
    ref = ref.relu()
    ybuf = plan.act(B, T, H, W, cout + (cout if slice_out else 0))
    ybuf.fill_(7.0)
    y = ybuf[..., cout:] if slice_out else ybuf
    plan.conv(x, y, w.double(), bias.double(), act=rt.ACT_RELU, res=res)
    plan.launch_all()
    torch.cuda.synchronize()
    err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
    assert err <= 2e-3 * max(ref.abs().max().item(), 1e-3), err
    if slice_out:
        assert (ybuf[..., :cout].float() == 7.0).all()


@pytest.mark.parametrize("ca,cb,groups", [(24, 24, 2), (240, 0, 3), (6, 6, 2), (3, 3, 2), (27, 27, 2), (12, 0, 3),
                                          (116, 116, 2), (15, 0, 3)])
def test_shuffle_concat(esf_lib, ca, cb, groups):
    """channel_shuffle(cat(a, b), groups) (shufflenetv2_helper.py:32-43, shufflenet_helper.py:24-34), bit exact;
    covers the 16/8/4-byte store variants and the scalar tail kernel."""
    g = torch.Generator().manual_seed(ca * 7 + cb)
    B, T, H, W = 2, 3, 5, 6
    plan = Plan(DEV, "fp16")
    a = plan.act(B, T, H, W, ca)
    a.copy_(_rand_act(g, B, T, H, W, ca, dtype=torch.float16))
    b = None
    if cb:
        bbuf = plan.act(B, T, H, W, cb + 8)       # second operand as a channel slice
        b = bbuf[..., 8:]
        b.copy_(_rand_act(g, B, T, H, W, cb, dtype=torch.float16))
    C = ca + cb
    y = plan.act(B, T, H, W, C)
    plan.shuffle_concat(a, b, groups, y)
    plan.launch_all()
    torch.cuda.synchronize()
    cat = torch.cat([a] + ([b] if cb else []), dim=4)
    ref = cat.reshape(B, T, H, W, groups, C // groups).transpose(4, 5).reshape(B, T, H, W, C)
    assert torch.equal(y.cpu(), ref.cpu())


@pytest.mark.parametrize("kt,cout", [(1, 64), (5, 8), (3, 6)])
def test_stem_conv(esf_lib, kt, cout):
    g = torch.Generator().manual_seed(kt)
    x = torch.randn(2, 3, 8, 32, 32, generator=g)
    k = (kt, 7, 7)
    w = torch.randn(cout, 3, *k, generator=g) * 0.1
    bias = torch.randn(cout, generator=g) * 0.1
    ref = F.conv3d(x, w, bias, (1, 2, 2), (kt // 2, 3, 3)).relu()
    y = torch.empty(_to_ndhwc(ref).shape, dtype=torch.bfloat16, device=DEV)
    plan = Plan(DEV)
    xd = x.to(DEV)
    plan.stem_conv(xd, y, w.double(), bias.double(), (1, 2, 2), (kt // 2, 3, 3))
    plan.launch_all()
    torch.cuda.synchronize()
    err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
    assert err <= 6e-3 * ref.abs().max().item()   # FP32 math, BF16 output rounding (2^-8 relative worst case)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("kt,cout,k,size", [(1, 64, 7, 64), (5, 8, 7, 64), (3, 24, 3, 48), (1, 64, 7, 224)])
def test_stem_banded_gemm(esf_lib, kt, cout, k, size, precision):
    """Tensor-core stem (banded implicit GEMM; the temporal-band kernel has its own test below) vs F.conv3d on the
    16-bit-rounded clip and weights."""
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(kt + cout)
    B, T = (2, 8) if size < 200 else (1, 2)
    x = torch.randn(B, 3, T, size, size, generator=g)
    kk = (kt, k, k)
    w = torch.randn(cout, 3, *kk, generator=g) * 0.1
    bias = torch.randn(cout, generator=g) * 0.1
    pad = (kt // 2, k // 2, k // 2)
    ref = F.conv3d(x.to(adt).float(), w.to(adt).float(), bias, (1, 2, 2), pad).relu()
    y = torch.full(_to_ndhwc(ref).shape, 7.0, dtype=adt, device=DEV)
    plan = Plan(DEV, precision)
    xd = x.to(DEV)
    pitch, lpad, _ = stem_route(xd.shape, w.shape, (1, 2, 2), pad)
    plan.stem_gemm(xd, y, w.double(), bias.double(), (1, 2, 2), pad, rt.ACT_RELU, pitch, lpad, 0)
    assert plan.meta[-1]["kind"] == "stem_igemm" and plan.meta[-1]["label"].endswith("banded")
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(y.cpu())
    err = (got - ref).abs().max().item()
    if not err <= 1e-2 * ref.abs().max().item():
        _diagnose("stem_banded", got, ref, 1e-2 * ref.abs().max().item())
    assert err <= 1e-2 * ref.abs().max().item()


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("B,cin,T,size,kt,cout", [
    (2, 3, 8, 64, 5, 8),       # the fast stem's geometry, one wave
    (3, 3, 21, 48, 5, 8),      # more frames than TMEM slots (ring re-use), odd batch (clipped box)
    (2, 3, 2, 64, 5, 8),       # fewer frames than time taps
    (1, 3, 1, 64, 5, 8),       # one frame: every slot is opened and published in the same step
    (2, 1, 6, 64, 5, 8),       # grey-scale clip (one 16-element K step)
    (2, 3, 6, 64, 3, 16),      # kT = 3, 64-column slots (8 slots)
    (2, 3, 5, 64, 5, 4),       # 16-column slots (32 slots)
    (8, 3, 4, 224, 5, 8),      # 196 tiles on 148 SMs: slots and stages carried from one tile into the next
])
def test_stem_temporal_band(esf_lib, B, cin, T, size, kt, cout, precision):
    """stem_tband_kernel (time taps folded into N, input frames streaming past a resident M tile, output frames in a ring
    of TMEM slots) vs F.conv3d on the 16-bit-rounded clip and weights, and bit-identical to nothing less than itself on a
    second launch (the barriers' phases must survive re-launching the same op)."""
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(B + T + cout)
    x = torch.randn(B, cin, T, size, size, generator=g)
    kk = (kt, 7, 7)
    w = torch.randn(cout, cin, *kk, generator=g) * 0.1
    bias = torch.randn(cout, generator=g) * 0.1
    pad = (kt // 2, 3, 3)
    assert rt.stem_tband_wb(size, cin, cout, kt, 7, 7, 2, 3) == 4
    ref = F.conv3d(x.to(adt).float(), w.to(adt).float(), bias, (1, 2, 2), pad).relu()
    y = torch.full(_to_ndhwc(ref).shape, 7.0, dtype=adt, device=DEV)
    plan = Plan(DEV, precision)
    xd = x.to(DEV)
    plan.stem(xd, y, w.double(), bias.double(), (1, 2, 2), pad)
    assert plan.meta[-1]["kind"] == "stem_igemm" and plan.meta[-1]["label"].endswith("t-band")
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(y.cpu())
    tol = 1e-2 * ref.abs().max().item()
    err = (got - ref).abs().max().item()
    if not err <= tol:
        _diagnose("stem_tband", got, ref, tol)
    assert err <= tol
    y.fill_(7.0)
    plan.launch_all()
    torch.cuda.synchronize()
    assert torch.equal(_to_ncdhw(y.cpu()), got)


def test_stem_temporal_band_random_geometries(esf_lib):
    """Seeded sweep over clip sizes the fixed cases do not hit: odd frame counts around the slot ring (15 .. 18, 33),
    batches that do not fill the 8-clip box, heights that leave a ragged last row tile, padded / unpadded time."""
    import random
    rnd = random.Random(7)
    done = 0
    for _ in range(40):
        B, T = rnd.choice([1, 2, 3, 5, 9]), rnd.choice([3, 7, 15, 16, 17, 18, 33])
        H, W = rnd.choice([40, 56, 72, 104]), rnd.choice([32, 64, 96])
        cin, cout, kt = rnd.choice([1, 3]), rnd.choice([4, 8, 16]), rnd.choice([3, 5])
        pt = rnd.choice([kt // 2, 0]) if T >= kt else kt // 2
        if rt.stem_tband_wb(W, cin, cout, kt, 7, 7, 2, 3) == 0 or B * T * H * W > 3_000_000:
            continue
        g = torch.Generator().manual_seed(done)
        x = torch.randn(B, cin, T, H, W, generator=g)
        w = torch.randn(cout, cin, kt, 7, 7, generator=g) * 0.1
        bias = torch.randn(cout, generator=g) * 0.1
        ref = F.conv3d(x.half().float(), w.half().float(), bias, (1, 2, 2), (pt, 3, 3)).relu()
        y = torch.full(_to_ndhwc(ref).shape, 7.0, dtype=torch.float16, device=DEV)
        plan = Plan(DEV, "fp16")
        plan.stem(x.to(DEV), y, w.double(), bias.double(), (1, 2, 2), (pt, 3, 3))
        assert plan.meta[-1]["label"].endswith("t-band")
        plan.launch_all()
        torch.cuda.synchronize()
        err = (_to_ncdhw(y.cpu()) - ref).abs().max().item()
        assert err <= 1e-2 * ref.abs().max().item(), (B, cin, T, H, W, cout, kt, pt, err)
        done += 1
        if done == 14:
            break
    assert done >= 10


def test_stem_temporal_band_matches_banded_stem(esf_lib):
    """Both tensor-core stems accumulate the same FP16 products in FP32: their outputs may differ only by the order of
    the additions (one 16-bit ulp at most after rounding)."""
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 3, 8, 64, 64, generator=g)
    w = torch.randn(8, 3, 5, 7, 7, generator=g) * 0.1
    bias = torch.randn(8, generator=g) * 0.1
    pitch, lpad, twb = stem_route(x.shape, w.shape, (1, 2, 2), (2, 3, 3))
    assert twb > 0
    outs = []
    for wb, label in ((twb, "t-band"), (0, "banded")):
        y = torch.empty(2, 8, 32, 32, 8, dtype=torch.float16, device=DEV)
        plan = Plan(DEV, "fp16")
        plan.stem_gemm(x.to(DEV), y, w.double(), bias.double(), (1, 2, 2), (2, 3, 3), rt.ACT_RELU, pitch, lpad, wb)
        assert plan.meta[-1]["label"].endswith(label)
        plan.launch_all()
        torch.cuda.synchronize()
        outs.append(y.float().cpu())
    assert (outs[0] - outs[1]).abs().max().item() <= 2 ** -10 * outs[1].abs().max().item()


@pytest.mark.parametrize("C", [64, 8, 6])
def test_pool3d(esf_lib, C):
    g = torch.Generator().manual_seed(C)
    x = _rand_act(g, 2, 4, 17, 18, C).to(DEV)
    for kernel, stride, pad, avg in [((1, 3, 3), (1, 2, 2), (0, 1, 1), False), ((3, 3, 3), (1, 2, 2), (1, 1, 1), False),
                                     ((1, 3, 3), (1, 2, 2), (0, 1, 1), True)]:
        xr = _to_ncdhw(x.cpu())
        ref = F.avg_pool3d(xr, kernel, stride, pad) if avg else F.max_pool3d(xr, kernel, stride, pad)
        y = torch.empty(_to_ndhwc(ref).shape, dtype=torch.bfloat16, device=DEV)
        plan = Plan(DEV)
        plan.pool(x, y, kernel, stride, pad, is_avg=avg)
        plan.launch_all()
        torch.cuda.synchronize()
        got = _to_ncdhw(y.cpu())
        if avg:
            assert (got - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()
        else:
            assert torch.equal(got, ref)   # max of BF16 values is exact


@pytest.mark.parametrize("C,off", [(30, 0), (19, 0), (60, 16), (243, 8), (9, 24)])
def test_pool3d_odd_channels_padded_rows(esf_lib, C, off):
    """C % 8 != 0 over rows with a 16-byte aligned pitch (the allocator's padding, or a slice of a concat buffer at a
    multiple of 8 channels): full groups of 8 channels vectorised, the ragged tail element-wise -- the neighbours of the
    slice and the row padding stay untouched."""
    g = torch.Generator().manual_seed(C + off)
    plan = Plan(DEV, "fp16")
    x = plan.act(2, 3, 13, 11, C)
    x.copy_(_rand_act(g, 2, 3, 13, 11, C, dtype=torch.float16))
    for kernel, stride, pad, avg in [((3, 3, 3), (1, 2, 2), (1, 1, 1), True), ((1, 3, 3), (1, 2, 2), (0, 1, 1), False),
                                     ((3, 3, 3), (2, 2, 2), (1, 1, 1), False)]:
        xr = _to_ncdhw(x.cpu())
        ref = F.avg_pool3d(xr, kernel, stride, pad) if avg else F.max_pool3d(xr, kernel, stride, pad)
        Bo, To, Ho, Wo, _ = _to_ndhwc(ref).shape
        ybuf = plan.act(Bo, To, Ho, Wo, off + C + 5)
        full = next(t for t in reversed(plan.keep) if isinstance(t, torch.Tensor))   # the padded allocation behind ybuf
        full.fill_(7.0)
        y = ybuf[..., off:off + C]
        plan.pool(x, y, kernel, stride, pad, is_avg=avg)
        plan.launch_all()
        torch.cuda.synchronize()
        got = _to_ncdhw(y.cpu())
        if avg:
            assert (got - ref).abs().max().item() <= 2e-3 * ref.abs().max().item()
        else:
            assert torch.equal(got, ref)
        assert (full[..., :off].float() == 7.0).all() and (full[..., off + C:].float() == 7.0).all()


@pytest.mark.parametrize("C,alpha", [(8, 4), (32, 4), (128, 4), (6, 4), (64, 8)])
def test_eca_fuse(esf_lib, C, alpha):
    g = torch.Generator().manual_seed(C)
    B, T, H, W = 2, 8, 9, 7
    xbuf = _rand_act(g, B, T, H, W, 2 * C).to(DEV)
    x = xbuf[..., C:]
    bn = torch.nn.BatchNorm3d(C)
    bn.weight.data = torch.rand(C, generator=g) + 0.5
    bn.bias.data = torch.rand(C, generator=g) - 0.5
    bn.running_mean = torch.randn(C, generator=g) * 0.3
    bn.running_var = torch.rand(C, generator=g) + 0.5
    bn.eval()
    wk = torch.rand(1, 1, 3, generator=g) - 0.5
    xr = _to_ncdhw(x.cpu())
    f = F.max_pool3d(xr, (alpha, 1, 1), (alpha, 1, 1))
    s = torch.sigmoid(F.conv1d(f.mean((2, 3, 4)).unsqueeze(1), wk, padding=1).squeeze(1))
    with torch.no_grad():
        ref = bn(f * s[:, :, None, None, None]).relu()
    ybuf = torch.zeros(B, T // alpha, H, W, 3 * C, dtype=torch.bfloat16, device=DEV)
    plan = Plan(DEV)
    plan.eca_fuse(x, ybuf[..., 2 * C:], alpha, wk, bn)
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(ybuf[..., 2 * C:].cpu())
    assert (got - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()
    assert (ybuf[..., :2 * C] == 0).all()


@pytest.mark.parametrize("C,off", [(60, 240), (120, 480), (240, 16), (20, 8), (9, 0)])
def test_eca_fuse_any_channel_count(esf_lib, C, off):
    """ECA fuse on the 16-byte path for channel counts that are not powers of two / not multiples of 8 (ShuffleNet's
    60 / 120 / 240): padded fast rows, output slice of a padded concat buffer; its neighbours stay untouched."""
    g = torch.Generator().manual_seed(C)
    B, T, H, W, alpha = 2, 8, 9, 7, 4
    plan = Plan(DEV, "fp16")
    x = plan.act(B, T, H, W, C)
    x.copy_(_rand_act(g, B, T, H, W, C, dtype=torch.float16))
    bn = torch.nn.BatchNorm3d(C)
    bn.weight.data = torch.rand(C, generator=g) + 0.5
    bn.bias.data = torch.rand(C, generator=g) - 0.5
    bn.running_mean = torch.randn(C, generator=g) * 0.3
    bn.running_var = torch.rand(C, generator=g) + 0.5
    bn.eval()
    wk = torch.rand(1, 1, 3, generator=g) - 0.5
    xr = _to_ncdhw(x.cpu()).float()
    f = F.max_pool3d(xr, (alpha, 1, 1), (alpha, 1, 1))
    s = torch.sigmoid(F.conv1d(f.mean((2, 3, 4)).unsqueeze(1), wk, padding=1).squeeze(1))
    with torch.no_grad():
        ref = bn(f * s[:, :, None, None, None]).relu()
    ybuf = plan.act(B, T // alpha, H, W, off + C + 3)
    full = next(t for t in reversed(plan.keep) if isinstance(t, torch.Tensor))
    full.fill_(7.0)
    y = ybuf[..., off:off + C]
    plan.eca_fuse(x, y, alpha, wk, bn)
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(y.cpu()).float()
    assert (got - ref).abs().max().item() <= 3e-3 * ref.abs().max().item()
    assert (full[..., :off].float() == 7.0).all() and (full[..., off + C:].float() == 7.0).all()


def _attention_reference(proj, B, T, H, W, d, gamma, scale, shift, alpha):
    N = T * H * W
    p = proj.double().reshape(B, N, 4, d)
    xd, q, k, v = p[:, :, 0], p[:, :, 1], p[:, :, 2], p[:, :, 3]
    att = torch.softmax(q @ k.transpose(1, 2), dim=-1)
    o = gamma * (att @ v) + xd
    o = (o * scale.double() + shift.double()).relu().reshape(B, T, H, W, d)
    return o.repeat_interleave(alpha, dim=1)


@pytest.mark.parametrize("d,T,H,W,qk_scale", [(8, 2, 9, 8, 1.0), (8, 2, 9, 8, 4.0), (8, 2, 16, 16, 4.0),
                                              (32, 2, 12, 11, 1.0), (32, 4, 8, 8, 2.0), (32, 4, 16, 8, 2.0),
                                              (64, 2, 7, 7, 1.0), (128, 2, 7, 7, 0.5), (16, 1, 9, 9, 1.0),
                                              (3, 2, 8, 8, 1.0), (12, 1, 20, 20, 1.0), (24, 2, 14, 14, 1.0),
                                              (32, 8, 14, 14, 1.0)])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_attention_tcgen05(esf_lib, d, T, H, W, qk_scale, precision):
    """tcgen05/TMEM fused attention vs FP64 softmax attention on the same FP32 projections."""
    adt = rt.TORCH_DTYPE[precision]
    g = torch.Generator().manual_seed(d + T)
    B, alpha = 2, 4
    N = T * H * W
    proj = torch.randn(B * N, 4 * d, generator=g)
    proj[:, d:3 * d] *= qk_scale / d ** 0.25
    gamma = 0.7
    scale = torch.rand(d, generator=g) + 0.5
    shift = torch.rand(d, generator=g) - 0.5
    ref = _attention_reference(proj, B, T, H, W, d, gamma, scale, shift, alpha)
    L = esf_lib
    nbytes = L.esf_attn_tc_pack_bytes(B, N, d)
    assert nbytes > 0
    packed = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    pj = proj.to(DEV)
    cpad = (2 * d + 7) // 8 * 8
    ybuf = torch.zeros(B, T * alpha, H, W, cpad, dtype=adt, device=DEV)
    yv = rt.view(ybuf[..., :d])
    sc, sh = scale.to(DEV), shift.to(DEV)
    s = rt.current_stream_ptr()
    h = ctypes.c_void_p()
    rt.check(L.esf_attn_tc_pack(pj.data_ptr(), B, N, d, rt.dtype_code(adt), packed.data_ptr(), s))
    rt.check(L.esf_attn_tc_create(packed.data_ptr(), B, T, H, W, d, gamma, sc.data_ptr(), sh.data_ptr(), alpha,
                                  ctypes.byref(yv), ctypes.byref(h)))
    rt.check(L.esf_op_launch(h, s))
    torch.cuda.synchronize()
    L.esf_op_destroy(h)
    got = ybuf[..., :d].cpu().double()
    err = (got - ref).abs().max().item()
    print("attn_tc %s d=%d N=%d rel err %.3e" % (precision, d, N, err / ref.abs().max().item()))
    tol = 1.5e-2 if precision == "bf16" else 3e-3   # P, V and the output are rounded to the storage format
    assert err <= tol * ref.abs().max().item(), "d=%d err %.4g scale %.4g" % (d, err, ref.abs().max().item())
    assert (ybuf[..., d:] == 0).all()


def test_attention_generic_fallback(esf_lib):
    d, T, H, W, B, alpha = 240, 2, 4, 5, 2, 4
    g = torch.Generator().manual_seed(3)
    N = T * H * W
    proj = torch.randn(B * N, 4 * d, generator=g)
    proj[:, d:3 * d] *= 1.0 / d ** 0.25
    scale = torch.rand(d, generator=g) + 0.5
    shift = torch.rand(d, generator=g) - 0.5
    ref = _attention_reference(proj, B, T, H, W, d, 0.7, scale, shift, alpha)
    ybuf = torch.zeros(B, T * alpha, H, W, 2 * d, dtype=torch.bfloat16, device=DEV)
    yv = rt.view(ybuf[..., :d])
    pj, sc, sh = proj.to(DEV), scale.to(DEV), shift.to(DEV)
    rt.check(esf_lib.esf_attn_generic(pj.data_ptr(), B, T, H, W, d, 0.7, sc.data_ptr(), sh.data_ptr(), alpha,
                                      ctypes.byref(yv), rt.current_stream_ptr()))
    torch.cuda.synchronize()
    got = ybuf[..., :d].cpu().double()
    assert (got - ref).abs().max().item() <= 6e-3 * ref.abs().max().item()   # FP32 math, BF16 output rounding
    assert (ybuf[..., d:] == 0).all()


def test_channel_plumbing_kernels(esf_lib):
    """shuffle-concat, elementwise add, SE channel scale, avg-pool + ReLU: bit-level semantics vs torch on BF16 data."""
    g = torch.Generator().manual_seed(11)
    B, T, H, W = 2, 3, 5, 7
    a = _rand_act(g, B, T, H, W, 9).to(DEV)
    b = _rand_act(g, B, T, H, W, 6).to(DEV)
    plan = Plan(DEV)
    ybuf = torch.zeros(B, T, H, W, 20, dtype=torch.bfloat16, device=DEV)
    plan.shuffle_concat(a, b, 3, ybuf[..., 2:17])
    y2 = torch.zeros(B, T, H, W, 9, dtype=torch.bfloat16, device=DEV)
    plan.shuffle_concat(a, None, 3, y2)
    a2 = _rand_act(g, B, T, H, W, 9).to(DEV)
    y3 = torch.zeros(B, T, H, W, 9, dtype=torch.bfloat16, device=DEV)
    plan.eltwise_add(a, a2, y3, act=rt.ACT_RELU)
    plan.launch_all()
    torch.cuda.synchronize()

    def shuffle(x, groups):   # NCDHW reference semantics (shufflenetv2_helper.py:32-43)
        bb, c, t, h, w = x.shape
        return x.view(bb, groups, c // groups, t, h, w).permute(0, 2, 1, 3, 4, 5).reshape(bb, c, t, h, w)
    ref = shuffle(torch.cat([_to_ncdhw(a.cpu()), _to_ncdhw(b.cpu())], 1), 3)
    assert torch.equal(_to_ncdhw(ybuf[..., 2:17].cpu()), ref)
    assert (ybuf[..., :2] == 0).all() and (ybuf[..., 17:] == 0).all()
    assert torch.equal(_to_ncdhw(y2.cpu()), shuffle(_to_ncdhw(a.cpu()), 3))
    assert torch.equal(y3.cpu().float(), (a.cpu().float() + a2.cpu().float()).relu().bfloat16().float())
    # squeeze-excite
    C, R = 12, 4
    x = _rand_act(g, B, T, H, W, C).to(DEV)
    se = torch.nn.Module()
    se.conv_reduce = torch.nn.Conv3d(C, R, 1)
    se.conv_expand = torch.nn.Conv3d(R, C, 1)
    y = torch.zeros_like(x)
    plan = Plan(DEV)
    plan.squeeze_excite(x, y, se)
    plan.pool(x, torch.zeros(B, T, 3, 4, C, dtype=torch.bfloat16, device=DEV), (1, 3, 3), (1, 2, 2), (0, 1, 1),
              is_avg=True, act=rt.ACT_RELU)
    plan.launch_all()
    torch.cuda.synchronize()
    xr = _to_ncdhw(x.cpu())
    with torch.no_grad():
        gate = F.relu6(se.conv_expand(F.relu(se.conv_reduce(xr.mean((2, 3, 4), keepdim=True)))) + 3.0) / 6.0
    ref = xr * gate
    assert (_to_ncdhw(y.cpu()) - ref).abs().max().item() <= 8e-3 * ref.abs().max().item()
    pooled = plan.keep[-1]


def test_head(esf_lib):
    g = torch.Generator().manual_seed(9)
    B = 3
    x0 = _rand_act(g, B, 2, 3, 3, 128).to(DEV)
    x1 = _rand_act(g, B, 8, 3, 3, 24).to(DEV)
    w = torch.randn(27, 152, generator=g) * 0.2
    b = torch.randn(27, generator=g) * 0.1
    feat = torch.cat([x0.cpu().float().mean((1, 2, 3)), x1.cpu().float().mean((1, 2, 3))], 1)
    logits = feat @ w.t() + b
    for act, ref in [(rt.HEAD_SOFTMAX, torch.softmax(logits, 1)), (rt.HEAD_NONE, logits), (rt.HEAD_RELU, logits.relu())]:
        plan = Plan(DEV)
        out = plan.head([x0, x1], w, b, act)
        plan.launch_all()
        torch.cuda.synchronize()
        assert (out.cpu() - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())


def test_errors_are_reported_not_swallowed(esf_lib):
    """bad arguments return an error code + message (no exception crosses the C boundary, no silent fallback)."""
    L = esf_lib
    x = torch.zeros(1, 2, 4, 4, 12, dtype=torch.bfloat16, device=DEV)   # stride 12 elements = 24 B: not 16 B aligned
    y = torch.zeros(1, 2, 4, 4, 16, dtype=torch.bfloat16, device=DEV)
    plan = Plan(DEV)
    with pytest.raises(rt.EsfError):
        plan.conv_igemm(x, y, torch.zeros(16, 12, 1, 1, 1).double(), torch.zeros(16).double())
    assert "multiple of 16" in L.esf_last_error().decode()


# ------------------------------------------------------------------------------------------------ Nonlocal block
@pytest.mark.parametrize("mode,n", [(0, 1568), (1, 392), (0, 37)])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_row_softmax(esf_lib, mode, n, dt):
    g = torch.Generator().manual_seed(21)
    rows, pitch = 300, (n + 3) // 4 * 4
    S = (torch.randn(rows, pitch, generator=g) * 3).to(DEV)
    ppitch = (n + 7) // 8 * 8
    P = torch.zeros(rows, ppitch, dtype=dt, device=DEV)
    scale = 0.0625 if mode == 0 else 1.0 / n
    rt.check(esf_lib.esf_row_softmax(S.data_ptr(), rows, n, pitch, scale, mode, rt.dtype_code(dt), P.data_ptr(), ppitch,
                                     rt.current_stream_ptr()))
    torch.cuda.synchronize()
    ref = torch.softmax(S[:, :n].double() * scale, dim=1) if mode == 0 else S[:, :n].double() * scale
    tol = 2 ** -10 if dt == torch.float16 else 2 ** -7
    assert ((P[:, :n].double() - ref).abs() <= tol * ref.abs() + 1e-7).all()
    assert (P[:, n:] == 0).all()


def test_transpose16(esf_lib):
    g = torch.Generator().manual_seed(22)
    B, rows, cols = 3, 100, 72
    x = torch.randn(B, rows, cols, generator=g).to(torch.float16).to(DEV)
    out = torch.zeros(B, 80, 128, dtype=torch.float16, device=DEV)
    rt.check(esf_lib.esf_transpose16(x.data_ptr(), B, rows, cols, rows * cols, cols, out.data_ptr(), 80 * 128, 128,
                                     rt.current_stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(out[:, :cols, :rows], x.transpose(1, 2))
    assert (out[:, cols:] == 0).all() and (out[:, :, rows:] == 0).all()


@pytest.mark.parametrize("inst,pool,group", [("softmax", [1, 2, 2], 1), ("dot_product", [1, 2, 2], 1),
                                             ("softmax", [1, 1, 1], 2)])
def test_nonlocal_block(esf_lib, inst, pool, group):
    """Plan.nonlocal_block vs the oracle's restatement of Nonlocal.forward on FP16-rounded operands."""
    from efficient_slowfast_b200.nets_resnet import Nonlocal
    from oracle import slowfast_oracle as O

    torch.manual_seed(5)
    B, T, H, W, C = 2, 4, 8, 8, 128
    nln = Nonlocal(C, C // 2, pool, instantiation=inst).eval()
    with torch.no_grad():
        for m in (nln.conv_theta, nln.conv_phi, nln.conv_g, nln.conv_out):
            m.weight.normal_(0, (2.0 / m.out_channels) ** 0.5)
            m.bias.uniform_(-0.1, 0.1)
        nln.bn.weight.uniform_(0.5, 1.5)
        nln.bn.bias.uniform_(-0.2, 0.2)
        nln.bn.running_mean.uniform_(-0.1, 0.1)
        nln.bn.running_var.uniform_(0.5, 1.5)
    x = torch.randn(B, T, H, W, C).to(torch.float16)
    plan = Plan(torch.device(DEV), precision="fp16")
    xd = x.to(DEV)
    y = torch.zeros_like(xd)
    with torch.no_grad():
        plan.nonlocal_block(xd, y, nln, group=group)
    plan.launch_all()
    torch.cuda.synchronize()
    sd = {"n." + k: v for k, v in nln.state_dict().items()}
    xr = _to_ncdhw(x).double()
    b, c, t, h, w = xr.shape
    if group > 1:
        xr = xr.permute(0, 2, 1, 3, 4).reshape(b * group, t // group, c, h, w).permute(0, 2, 1, 3, 4)
    ref = O.nonlocal_block(xr, {k: v.double() for k, v in sd.items()}, "n", pool, inst)
    if group > 1:
        ref = ref.permute(0, 2, 1, 3, 4).reshape(b, t, c, h, w).permute(0, 2, 1, 3, 4)
    got = _to_ncdhw(y.cpu()).double()
    err = ((got - ref).abs().max() / ref.abs().max()).item()
    print("nonlocal %s pool %s group %d: rel err %.3e" % (inst, pool, group, err))
    assert err < 1e-2


@pytest.mark.parametrize("C,shape", [(72, (2, 8, 28, 28)), (960, (3, 4, 7, 7)), (12, (2, 16, 14, 14)), (240, (1, 32, 56, 56))])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_global_mean(esf_lib, C, shape, dt):
    """esf_global_mean (two-pass, deterministic) vs torch.mean on the 16-bit-rounded activation, inside a wider row."""
    B, T, H, W = shape
    g = torch.Generator().manual_seed(C)
    Cp = (C + 7) // 8 * 8 if C >= 8 else C
    xbuf = _rand_act(g, B, T, H, W, Cp, dtype=dt).to(DEV)
    x = xbuf[..., :C]
    feat = torch.full((B, C + 5), 7.0, device=DEV)
    scratch = torch.empty(int(esf_lib.esf_global_mean_scratch_floats(B, C)), device=DEV)
    xv = rt.view(x)
    for _ in range(2):
        rt.check(esf_lib.esf_global_mean(ctypes.byref(xv), scratch.data_ptr(), feat.data_ptr(), C + 5, 3,
                                         rt.current_stream_ptr()))
    torch.cuda.synchronize()
    ref = x.float().mean(dim=(1, 2, 3))
    assert torch.allclose(feat[:, 3:3 + C], ref, rtol=1e-4, atol=1e-5)
    assert (feat[:, :3] == 7.0).all() and (feat[:, 3 + C:] == 7.0).all()
    first = feat.clone()
    rt.check(esf_lib.esf_global_mean(ctypes.byref(xv), scratch.data_ptr(), feat.data_ptr(), C + 5, 3, rt.current_stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(first, feat)            # deterministic


@pytest.mark.parametrize("cin,W,kw,pw", [(3, 224, 7, 3), (3, 64, 7, 3), (1, 112, 7, 3), (3, 48, 3, 1), (2, 40, 5, 2),
                                         (3, 50, 7, 3)])
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_stem_pack_variants(esf_lib, cin, W, kw, pw, precision):
    """esf_stem_pack / _lo / _gather against a torch restatement of the packed row layout, for the shared-memory staged
    kernel (W % 4 == 0; the static 24-element path when Cin = 3) and the scalar-load kernel (W = 50)."""
    adt = rt.TORCH_DTYPE[precision]
    geo = rt.stem_geometry(W, cin, kw, 2, pw)
    if geo is None:
        pytest.skip("no banded geometry")
    pitch, lpad, _ = geo
    g = torch.Generator().manual_seed(cin * W)
    B, T, H = 2, 6, 5
    x = (torch.randn(B, cin, T, H, W, generator=g) * 3).to(DEV)
    idx = torch.tensor([0, 2, 5], dtype=torch.int32, device=DEV)

    def expect(src, lo):
        rows = src.permute(0, 2, 3, 4, 1).reshape(B, src.shape[2], H, W * cin)        # (w, c) interleaved
        v = rows - rows.to(adt).float() if lo else rows
        out = torch.zeros(B, src.shape[2], H, pitch, device=DEV)
        out[..., lpad:lpad + W * cin] = v
        return out.to(adt)

    a = torch.full((B, T, H, pitch), 7.0, dtype=adt, device=DEV)
    rt.check(esf_lib.esf_stem_pack(x.data_ptr(), B, cin, T, H, W, pitch, lpad, rt.dtype_code(adt), a.data_ptr(), None))
    lo = torch.full((B, T, H, pitch), 7.0, dtype=adt, device=DEV)
    rt.check(esf_lib.esf_stem_pack_lo(x.data_ptr(), B, cin, T, H, W, pitch, lpad, rt.dtype_code(adt), lo.data_ptr(), None))
    ga = torch.full((B, 3, H, pitch), 7.0, dtype=adt, device=DEV)
    rt.check(esf_lib.esf_stem_pack_gather(x.data_ptr(), B, cin, T, H, W, idx.data_ptr(), 3, pitch, lpad,
                                          rt.dtype_code(adt), ga.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(a, expect(x, False))
    assert torch.equal(lo, expect(x, True))
    assert torch.equal(ga, expect(x.index_select(2, idx.long()), False))


def test_pool3d_fp16_packed_max(esf_lib):
    """The packed 16-bit max path (full 16-byte groups, max-pool, no activation) in FP16 with -inf padding semantics."""
    g = torch.Generator().manual_seed(5)
    x = _rand_act(g, 2, 3, 15, 14, 24, dtype=torch.float16).to(DEV)
    x[0, 0, 0, 0, :] = -60000.0          # a window whose only valid taps are very negative must not see the padding
    for kernel, stride, pad in [((1, 3, 3), (1, 2, 2), (0, 1, 1)), ((3, 3, 3), (1, 2, 2), (1, 1, 1)), ((2, 1, 1), (2, 1, 1), (0, 0, 0))]:
        ref = F.max_pool3d(_to_ncdhw(x.cpu()), kernel, stride, pad)
        y = torch.empty(_to_ndhwc(ref).shape, dtype=torch.float16, device=DEV)
        plan = Plan(DEV, "fp16")
        plan.pool(x, y, kernel, stride, pad)
        plan.launch_all()
        torch.cuda.synchronize()
        assert torch.equal(_to_ncdhw(y.cpu()), ref)


def test_position_attention_with_channel_reduction(esf_lib):
    """SpatialAttention(reduction = 2) (wdf_attention_helper.py:17-26; no cfg key of the reference reaches it): query / key
    with d / 2 channels run on the same kernels through zero-padded projection rows."""
    from efficient_slowfast_b200.nets_resnet import FuseFastAndSlow

    g = torch.Generator().manual_seed(9)
    B, T, H, W, C, beta, alpha = 2, 2, 6, 5, 64, 8, 4
    fuse = FuseFastAndSlow([C, C // beta], alpha, beta, torch.nn.BatchNorm3d, reduction=2)
    d = C // beta
    with torch.no_grad():
        for prm in fuse.parameters():
            prm.copy_(torch.randn(prm.shape, generator=g) * 0.3)
        fuse.attention_spatial_s2f.gamma.fill_(0.6)
        bn = fuse.bn_s2f
        bn.running_mean.copy_(torch.randn(d, generator=g) * 0.2)
        bn.running_var.copy_(torch.rand(d, generator=g) + 0.5)
    fuse.eval()
    att = fuse.attention_spatial_s2f
    assert att.query_conv.out_channels == d // 2
    x = torch.randn(B, C, T, H, W, generator=g)
    with torch.no_grad():    # wdf_attention_helper.py:33-54 + custom_video_model_builder.py:141-146, FP64
        xd = F.conv3d(x.double(), fuse.downsample_c_of_slow.weight.double())
        N = T * H * W
        q = F.conv3d(xd, att.query_conv.weight.double(), att.query_conv.bias.double()).view(B, -1, N).permute(0, 2, 1)
        k = F.conv3d(xd, att.key_conv.weight.double(), att.key_conv.bias.double()).view(B, -1, N)
        v = F.conv3d(xd, att.value_conv.weight.double(), att.value_conv.bias.double()).view(B, -1, N)
        o = torch.bmm(v, torch.softmax(torch.bmm(q, k), dim=-1).permute(0, 2, 1)).view(B, d, T, H, W)
        ref = bn.double()(att.gamma.double() * o + xd).relu().repeat_interleave(alpha, dim=2)
    bn.float()
    plan = Plan(DEV, "fp16")
    xs = plan.act(B, T, H, W, C)
    xs.copy_(_to_ndhwc(x).to(torch.float16))
    ybuf = plan.act(B, T * alpha, H, W, 2 * d)
    plan.position_attention(xs, ybuf[..., :d], alpha, fuse.downsample_c_of_slow.weight, att, bn)
    plan.launch_all()
    torch.cuda.synchronize()
    got = _to_ncdhw(ybuf[..., :d].cpu()).double()
    assert (got - ref).abs().max().item() <= 1e-2 * ref.abs().max().item()
